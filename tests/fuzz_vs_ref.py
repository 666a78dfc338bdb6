#!/usr/bin/env python3
"""Mutation fuzzer: a converter binary vs the reference gaf2paf on single malformed
or unusual records.  Compares exit code and stdout (and stderr text for rc 1).

    python tests/fuzz_vs_ref.py [--n 2000] [--seed 1] [--bin build/g2p_hostsim] [--long]

The reference is the unmodified build in oracle/_ref when present, else the restatement
oracle/bin/gaf2paf_oracle (tests/helpers.py oracle_path).  CIGAR text outside the SAM
grammar that std::stol accepts is handled like the reference does; the only tolerated class is
int64 overflow (undefined behaviour in the reference), see `tolerated()`.
"""
import argparse
import os
import random
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers as H  # noqa: E402

LENGTHS = "chrA\t1000\nchrB\t500\nchrC\t300\na\t10\nb\t5\nc\t10\nn2\t20\nn3\t50\nz\t0\naveryveryverylongname_12345\t77\n"

SEEDS = [
    "q1 200 5 132 + >chrA:100-200>chrB:0-50 150 10 138 120 130 60 tp:A:P cm:i:5 cg:Z:50M2I40M3D35M",
    "q1 200 5 132 - >chrA:100-200<chrB:0-50 150 10 138 120 130 0 cg:Z:50M2I40M3D35M",
    "q1 200 5 132 - chrC 300 10 138 120 130 60 rc:Z:foo tp:A:S cg:Z:50M2I40M3D35M",
    "q1 200 5 132 + >chrA:0-100<n2>n3 170 10 138 120 130 60 cg:Z:50M2I40M3D35M",
    "q 100 0 28 + >a>b>c 25 0 25 25 28 60 cg:Z:10M3I5M10M",
    "q 100 0 24 + >a>b>c 25 0 25 20 25 60 cg:Z:2S2H8M2N3P5M7M3X",
    "q 100 10 27 - >a<b>c 25 3 20 17 17 300 cg:Z:17M",
    "q 100 0 23 + >a>z>c 20 0 20 20 23 60 cg:Z:10M3I10M",
    "q 100 3 30 - >a<b>c 25 2 24 20 27 13 tp:A:P cg:Z:4M2I6M3D5M1I4M",
    "q 100 0 30 + <c<b<a 25 1 24 20 28 60 cg:Z:3M2I4M1D2M3I10M2D1M",
    "q 100 0 15 + >averyveryverylongname_12345:0-15 15 0 15 15 15 60 cg:Z:15M",
]

WEIRD = ["*", "", "-5", " 12", "+7", "12x", "x12", "99999999999999999999", "0", "1", "007", "-", "+", "255", "256",
         "9223372036854775807", "9223372036854775808", "\x0b3", "3 4"]
WEIRD_STEP = [">a", "<b", ">c:0-5", ">c:5", ">:0-5", ">>", "<", ">a:", ">a:-", ">a:1-", ">a:-3", ">a:1--3", ">nope",
              ">chrA:10-20", "chrB", "*", ">a:2-8x", ">a: 2-8", ">n2:0-20:9"]
WEIRD_CG = ["", "M", "5", "5M", "0M", "5Q", "5M3", "-5M", "+5M", " 5M", "5 M", "05M", "5m", "10=", "3X", "2I", "2D", "99999999999M",
            "5M\r", "1M1M1M1M", "20M", "3S", "4H", "2N", "1P", "-3M", "-2I", "5Q3M", "5.5M", "0005M", "00M", "9223372036854775807M",
            "9223372036854775808M", "-9223372036854775808D", "\t", "5 5M", "+0M", "x", "3=-1X", "7MM", "\x0b4M", "4M-", "--4M"]
TAGS = ["tp:A:P", "tp:A:S", "rc:Z:x", "rc:Z:", "cm:i:5", "ab:1", "abc", "a:b:c", "xx:Z:y:z", "tp:ZZ:hello", "cg:Z:5M", "", "tpp:A:P", ":::::", "cg:i:5M"]


def mutate(rnd, line):
    cols = line.split(" ")
    k = rnd.randrange(12)
    r = rnd.random()
    if r < 0.25:
        # numeric / any column <- weird value
        i = rnd.randrange(len(cols))
        cols[i] = rnd.choice(WEIRD)
    elif r < 0.45:
        # path surgery
        p = cols[5]
        toks = re.findall(r"[<>][^<>]*", p) or [p]
        op = rnd.randrange(4)
        if op == 0:
            toks[rnd.randrange(len(toks))] = rnd.choice(WEIRD_STEP)
        elif op == 1:
            toks.insert(rnd.randrange(len(toks) + 1), rnd.choice(WEIRD_STEP))
        elif op == 2 and len(toks) > 1:
            del toks[rnd.randrange(len(toks))]
        else:
            toks = [rnd.choice(WEIRD_STEP) for _ in range(rnd.randrange(1, 4))]
        cols[5] = "".join(toks)
    elif r < 0.65:
        # cigar surgery
        for i, c in enumerate(cols):
            if c.startswith("cg:Z:"):
                ops = re.findall(r"\d+[A-Z=]", c[5:])
                op = rnd.randrange(4)
                if op == 0 and ops:
                    ops[rnd.randrange(len(ops))] = rnd.choice(WEIRD_CG)
                elif op == 1:
                    ops.insert(rnd.randrange(len(ops) + 1), rnd.choice(WEIRD_CG))
                elif op == 2 and len(ops) > 1:
                    del ops[rnd.randrange(len(ops))]
                else:
                    ops = [rnd.choice(WEIRD_CG) for _ in range(rnd.randrange(0, 5))]
                cols[i] = "cg:Z:" + "".join(ops)
    elif r < 0.8:
        # tag surgery
        op = rnd.randrange(3)
        if op == 0:
            cols.insert(rnd.randrange(12, len(cols) + 1), rnd.choice(TAGS))
        elif op == 1 and len(cols) > 12:
            del cols[rnd.randrange(12, len(cols))]
        else:
            cols.append(rnd.choice(TAGS))
    elif r < 0.9:
        # drop / duplicate a column
        if rnd.random() < 0.5:
            del cols[k]
        else:
            cols.insert(k, cols[k])
    else:
        # coordinates tweak keeping syntax
        i = rnd.choice([2, 3, 7, 8, 9, 10, 11])
        if i < len(cols) and cols[i].isdigit():
            cols[i] = str(max(0, int(cols[i]) + rnd.randrange(-12, 13)))
    return "\t".join(cols)


def run(binary, lp, data):
    try:
        p = subprocess.run([binary, "-", "-l", lp], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=20)
    except subprocess.TimeoutExpired:
        return 999, b"", b"TIMEOUT"
    rc = p.returncode
    if rc < 0:
        rc = 128 - rc
    return rc, p.stdout, p.stderr


CG_STRICT = re.compile(rb"^(\d+[MIDNSHPX=])*$")


def tolerated(line, ref, got):
    """The one tolerated class: CIGAR lengths of 19 digits (|v| >= 10^18).  Their sums overflow
    int64, which is undefined behaviour in the reference (its outcome depends on how the compiler
    happened to arrange the arithmetic), so there is nothing to be identical to.  Everything else
    -- sign, blanks, trailing junk, negative or zero lengths -- must match exactly."""
    m = re.search(rb"\tcg:[^\t:]*:([^\t]*)", line)
    return bool(m and re.search(rb"\d{19,}", m.group(1)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--bin", default=os.path.join(ROOT, "build", "g2p_hostsim"))
    ap.add_argument("--long", action="store_true", help="append a 300-byte tag to every case: the records take the long-record kernels (k_par, k_long)")
    a = ap.parse_args()
    rnd = random.Random(a.seed)
    ref_bin, kind = H.oracle_path()
    bad = 0
    tol = 0
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "w").write(LENGTHS)
        for it in range(a.n):
            line = rnd.choice(SEEDS)
            for _ in range(rnd.randrange(1, 3)):
                line = mutate(rnd, line.replace("\t", " "))
            data = line.replace(" ", "\t") if "\t" not in line else line
            if a.long:
                data += "\tzy:Z:" + "p" * 300
            data = data.encode("latin-1") + b"\n"
            ref = run(ref_bin, lp, data)
            got = run(a.bin, lp, data)
            same = ref[0] == got[0] and (ref[0] == 134 or ref[1] == got[1]) and (ref[0] != 1 or ref[2] == got[2])
            if not same:
                if tolerated(data, ref, got):
                    tol += 1
                    continue
                bad += 1
                if bad <= 15:
                    print("MISMATCH #%d: %r" % (it, data))
                    print("   ref rc=%d out=%r err=%r" % (ref[0], ref[1][:200], ref[2][-160:]))
                    print("   got rc=%d out=%r err=%r" % (got[0], got[1][:200], got[2][-160:]))
    print("fuzz: %d cases, %d mismatches, %d tolerated (int64-overflow UB in the reference), %s oracle" % (a.n, bad, tol, kind))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
