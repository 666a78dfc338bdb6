#!/usr/bin/env python3
"""Mutation fuzzer for gaffilter: the filter kernels under the SIMT emulator (build/g2p_filter_simt) vs the reference
gaffilter on small inputs (a few query sequences, ~40 records) with one or two mutated records, random option sets, GAF and
PAF mode.  Compares the exit code, stdout and the "[gaffilter]: ..." summary line.  The checker is the reference build
(oracle/_ref/gaffilter) when present, else the restatement oracle/bin/gaffilter_oracle (tests/helpers.py oracle_path).

    python tests/fuzz_filter_vs_ref.py [--n 1000] [--seed 1]

Development tool; tests/test_filter_edges.py runs a few hundred of these cases."""
import argparse
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers as H
from fuzz_vs_ref import mutate

SIMT = os.path.join(ROOT, "build", "g2p_filter_simt")
OPTS = [["-r", "2"], ["-r", "5", "-m", "0.25"], ["-o", "100"], ["-r", "3", "-q", "5", "-b", "50"], ["-r", "2", "-o", "200", "-m", "0.1"], ["-r", "1.5", "-i", "1.01"]]


def run(cmd, data):
    try:
        p = subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=30)
    except subprocess.TimeoutExpired:
        return 999, b"", ""
    rc = p.returncode
    err = p.stderr.decode("latin-1").strip().split("\n")
    return (128 - rc if rc < 0 else rc), p.stdout, err[-1] if err else ""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    rnd = random.Random(a.seed)
    ref_bin, kind = H.oracle_path("auto", "gaffilter")
    bad = 0
    for it in range(a.n):
        paf = rnd.random() < 0.5
        text, _ = H.gen_filter_case(a.seed * 100000 + it, n_records=40, n_queries=rnd.choice([1, 3, 12]), paf=paf)
        lines = [l.decode("latin-1") for l in text.split(b"\n") if l]
        for _ in range(rnd.randrange(0, 3)):
            k = rnd.randrange(len(lines))
            lines[k] = mutate(rnd, lines[k].replace(" ", "\x01").replace("\t", " ")).replace("\x01", " ")
        data = ("\n".join(lines) + "\n").encode("latin-1")
        args = rnd.choice(OPTS) + (["-p"] if paf else [])
        ref = run([ref_bin] + args + ["-"], data)
        got = run([SIMT] + args + ["-"], data)
        same = ref[0] == got[0] and ref[1] == got[1] and (ref[0] != 0 or ref[2] == got[2])
        if not same:
            bad += 1
            if bad <= 10:
                print("MISMATCH #%d args=%s" % (it, args))
                for l in lines:
                    print("     " + repr(l))
                print("   ref rc=%d lines=%d err=%r" % (ref[0], ref[1].count(b"\n"), ref[2][-120:]))
                print("   got rc=%d lines=%d err=%r" % (got[0], got[1].count(b"\n"), got[2][-120:]))
    print("fuzz gaffilter: %d cases, %d mismatches, %s oracle" % (a.n, bad, kind))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
