"""gaf2paf's fast conversion kernels at their 32-bit limits, against the 64-bit reference.

The reference parses every number with std::stol and computes in int64.  The fast kernels (k_fuse, k_rec, k_short,
k_par_*, k_long) compute in 32 bits: each checks its inputs and hands a record it cannot take on to the next kernel of
the chain, down to the general per-record kernel (k_convert_list, int64 throughout).  These tests put numbers at and
just past every such limit and assert two things for every case in every configuration: the bytes (and exit code)
equal the reference's, and the record was converted by the kernel the configuration names, or handed on by it.
A case that quietly reached the general kernel would prove nothing about the fast one.

The limits (DESIGN.md §7, "numeric limits"):
  - numeric columns and ':start-end' bounds: at most 9 digits                 k_fuse, k_rec, k_short, k_par, k_long
  - lengths-table value: 0 <= len <= 2^31-1 (bit 31 is k_rec's / k_fuse's interval flag)
  - summed step length of a '-' record (flip_gaf's total): at most 2^31-1
  - CIGAR op: 1-7 digits (k_par keeps 24 bits of the length)
  - block-length sum of a record at most 2^31-1 (k_par: the query coordinate is a u32 up to ~3.15e9)
  - k_long: q0 + q, nm and nb of a line at most 2^31-1
  - gi:f: through the 0..1 fast formatter only; anything else is handed on

Configurations (CONFIGS): k_fuse (G2P_FUSE=2), k_rec (G2P_FUSE=0), k_short (G2P_SIZE_KERNEL=short), k_par (the record
padded past k_rec's 240 bytes with an extra tag), k_long (the same with G2P_PAR=0), and k_long on unpadded records
(build/g2p_simt_long, compiled with G2P_S_LIMIT=0, with G2P_PAR=0).  The CPU tests run the kernels under the SIMT
emulator; the GPU tests run the same cases through the C-ABI, the gaf2paf executable and the device-resident path."""
import math
import os
import random
import re
import subprocess
import tempfile

import pytest

import helpers as H

SIMT = os.path.join(H.BUILD, "g2p_simt")
SIMT_LONG = os.path.join(H.BUILD, "g2p_simt_long")
EXE = os.path.join(H.ROOT, "cactus-gfa-tools_b200", "bin", "gaf2paf")

I31 = 2 ** 31 - 1
PAD = "zz:Z:" + "x" * 240   # an extra tag: longer than k_rec's / k_short's 240 bytes, not printed

# ---- configurations: name -> (binary, environment, pad the case records) -----------------------------------------
CONFIGS = {
    "fuse": (SIMT, {"G2P_FUSE": "2"}, False),
    "rec": (SIMT, {"G2P_FUSE": "0"}, False),
    "short": (SIMT, {"G2P_FUSE": "0", "G2P_SIZE_KERNEL": "short"}, False),
    "par": (SIMT, {"G2P_FUSE": "0"}, True),
    "long": (SIMT, {"G2P_FUSE": "0", "G2P_PAR": "0"}, True),
    "slong": (SIMT_LONG, {"G2P_FUSE": "0", "G2P_PAR": "0"}, False),
}
ORDER = ("fuse", "rec", "short", "par", "long", "slong")


def gaf(qn, qlen, qs, qe, strand, path, ps, pe, m, b, cg, mapq=60, plen=None, tags=("tp:A:P",)):
    cols = [qn, qlen, qs, qe, strand, path, plen if plen is not None else 999, ps, pe, m, b, mapq]
    return "\t".join(str(c) for c in cols + list(tags) + ["cg:Z:" + cg])


# Ordinary records around every case: a wrong hand-off or a wrong output offset shows in them.
BASE_LENGTHS = "o1\t100\no2\t80\no3\t120\n"
ORDINARY = [
    gaf("ord1", 150, 10, 115, "+", ">o1", 0, 100, 98, 105, "50M5I50M"),
    gaf("ord2", 300, 20, 180, "-", ">o1<o2", 5, 170, 150, 170, "60M5D100M", mapq=30),
    gaf("ord3", 90, 0, 148, "+", ">o2:10-70>o3", 5, 150, 140, 148, "40M3I105M", tags=("tp:A:S", "rc:Z:x")),
    gaf("ord4", 500, 7, 107, "-", "<o3", 10, 110, 100, 100, "100M", mapq=255),
]


def batch(records, pad):
    if pad:
        records = [r.replace("\tcg:Z:", "\t" + PAD + "\tcg:Z:", 1) for r in records]
    lines = ORDINARY[:2] + [x for r in records for x in (r, ORDINARY[2])] + ORDINARY[3:]
    return ("\n".join(lines) + "\n").encode()


# ---- routes ------------------------------------------------------------------------------------------------------
_FUSED = re.compile(r"k_fuse converted (\d+) records")
_PIPE = re.compile(r"(\d+) records, (\d+) to k_par \((\d+) steps, (\d+) ops\), (\d+) to k_long, (\d+) to the general kernel")


def run_simt(binary, env, lp, data):
    """-> (exit code, stdout, route) with route = ("fused", n) or ("pipe", records, to_k_par, par_steps, to_k_long, general)."""
    e = dict(os.environ, G2P_SIMT_STATS="1", **env)
    p = subprocess.run([binary, "-l", lp, "-"], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e)
    rc = p.returncode if p.returncode >= 0 else 128 - p.returncode
    err = p.stderr.decode("latin-1")
    m = _FUSED.search(err)
    if m:
        return rc, p.stdout, ("fused", int(m.group(1)))
    m = _PIPE.search(err)
    assert m, err[-300:]
    g = [int(x) for x in m.groups()]
    return rc, p.stdout, ("pipe", g[0], g[1], g[2], g[4], g[5])


def route_of(cfg, st, nrec, k):
    """'F' if the configuration's fast kernel converted the k case records of a batch of nrec, 'H' if it handed them
    all on; anything else (some of them, or ordinary records handed on too) is returned as a description."""
    if cfg == "fuse":
        return "F" if st == ("fused", nrec) else ("H" if st[0] == "pipe" else repr(st))
    if st[0] != "pipe":
        return repr(st)
    _, n, to_par, steps, to_long, general = st
    if cfg in ("rec", "short"):
        return {0: "F", k: "H"}.get(to_par, repr(st))
    if cfg == "par":   # k_rec hands the padded records to k_par, which converts them or hands them to k_long
        if to_par != k:
            return repr(st)
        if to_long == 0 and steps > 0:
            return "F"
        return "H" if to_long == k else repr(st)   # (no steps: k_par's header pass rejected every record)
    want = k if cfg == "long" else nrec   # every record reaches k_long (g2p_simt_long: also the ordinary ones)
    if to_par != want or to_long != want:
        return repr(st)
    return {0: "F", k: "H"}.get(general, repr(st))


def oracle(lp, data):
    binary, _ = H.oracle_path("auto", "gaf2paf")
    return H.run_tool(binary, ["-", "-l", lp], data)


def check_case(td, lengths, records, routes, configs=ORDER):
    """Run `records` (between ordinary ones) in every configuration; `routes` is one letter per configuration of
    ORDER: F (the fast kernel converts them) or H (it hands them on)."""
    lp = os.path.join(td, "l.tsv")
    with open(lp, "w") as f:
        f.write(BASE_LENGTHS + lengths)
    want = dict(zip(ORDER, routes))
    bad = []
    for cfg in configs:
        binary, env, pad = CONFIGS[cfg]
        data = batch(records, pad)
        nrec = data.count(b"\n")
        rc, ref, err = oracle(lp, data)
        assert rc == 0 and ref.count(b"\n") >= 4, (cfg, err[-300:])
        grc, out, st = run_simt(binary, env, lp, data)
        if grc != rc or out != ref:
            bad.append("%s: bytes differ from the reference (exit %d, %d vs %d bytes)" % (cfg, grc, len(out), len(ref)))
            continue
        got = route_of(cfg, st, nrec, len(records))
        if got != want[cfg]:
            bad.append("%s: route %s, want %s" % (cfg, got, want[cfg]))
    return bad


# ---- the case table ----------------------------------------------------------------------------------------------
# Each case: (name, extra lengths TSV, [records], routes over ORDER = fuse rec short par long slong).
FAST, ON = "FFFFFF", "HHHHHH"
CASES = []


def case(name, lengths, records, routes):
    CASES.append((name, lengths, records if isinstance(records, list) else [records], routes))


# numeric columns 2-4 and 7-11 at the 9-digit limit and past it.  `big` is a node of 2^31-1 bases; nodes of other
# lengths are added where a column's value needs them.
COLVALS = [999999999, 1000000000, 2147483647, 2147483648, 4294967295, 4294967296, 9223372036854775807]
for col in ("qlen", "qs", "qe", "plen", "ps", "pe", "matches", "block"):
    for v in COLVALS:
        r = dict(qlen=150, qs=10, qe=110, ps=1000, pe=1095, m=95, b=100, plen=None)
        if col == "qs":   # the reference does not check qe against the CIGAR: qe stays at 9 digits
            r["qs"], r["qe"] = v, 999999999
        elif col == "matches":   # m <= b keeps gi:f: in 0..1
            r["m"] = r["b"] = v
        elif col == "ps":   # a window of 95 bases starting at v, on a node that holds it
            r["ps"], r["pe"] = (v, v + 95) if v + 95 < 2 ** 63 else (v - 95, v)
        elif col == "pe":
            r["ps"], r["pe"] = v - 95, v
        else:
            r[{"block": "b"}.get(col, col)] = v
        node = max(I31, r["pe"])
        fast = v == 999999999 and r["pe"] <= 999999999
        for strand in "+-":
            case("col-%s-%d%s" % (col, v, strand), "big\t%d\n" % node,
                 gaf("c" + col, r["qlen"], r["qs"], r["qe"], strand, ">big", r["ps"], r["pe"], r["m"], r["b"], "50M5I45M", plen=r["plen"]),
                 FAST if fast else ON)



# interval bounds of 9 and 10 digits, an empty interval, an interval ending at its node's length
for strand in "+-":
    case("ivl-9-digits" + strand, "big\t%d\n" % I31, gaf("iv", 150, 10, 115, strand, ">big:999999899-999999999", 0, 100, 95, 105, "50M5I50M"), FAST)
    case("ivl-10-digits" + strand, "big\t%d\n" % I31, gaf("iv", 150, 10, 115, strand, ">big:999999999-1000000099", 0, 100, 95, 105, "50M5I50M"), ON)
    case("ivl-start-is-end" + strand, "big\t%d\n" % I31, gaf("iv", 150, 10, 105, strand, ">o1>big:500-500<o2", 50, 140, 90, 95, "45M5I45M"), FAST)
    case("ivl-ends-at-node-length" + strand, "n9\t999999999\n", gaf("iv", 150, 10, 115, strand, "<n9:999999900-999999999", 0, 99, 95, 104, "50M5I49M"), FAST)
    case("ivl-ends-at-2^31-1" + strand, "big\t%d\n" % I31, gaf("iv", 150, 10, 115, strand, ">big:2147483547-2147483647", 0, 100, 95, 105, "50M5I50M"), ON)

# lengths-table values on '>' and '<' steps of '+' and '-' records
for L in (0, I31, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 33 + 7):
    for strand in "+-":
        for d in "><":
            if L == 0:   # a node of no bases inside the path
                rec = gaf("tl", 150, 10, 105, strand, ">o1%st<o2" % d, 50, 140, 90, 95, "45M5I45M")
            else:
                rec = gaf("tl", 150, 10, 110, strand, d + "t", 1000, 1095, 95, 100, "50M5I45M")
            case("table-%d%s%s" % (L, strand, d), "t\t%d\n" % L, rec, FAST if L <= I31 else ON)
        # stol accepts a negative length: it is printed as the target length of an interval step
        case("table-negative" + strand, "neg\t-5\n", gaf("tl", 150, 10, 155, strand, ">o1<neg:0-50>o2", 50, 190, 140, 145, "70M5I70M"), ON)

# '-' records: flip_gaf mirrors the window about the summed step lengths, which k_rec / k_fuse / k_par / k_long keep in
# 31 bits.  Two steps that cross 2^31 only together, and the same with interval steps; '+' records do not sum.
for total in (I31, 2 ** 31):
    t = "t\t%d\n" % (total - 100)
    for strand in "+-":
        # k_par sums the step lengths of '+' records too (32-bit prefix sums of its step table)
        rt = FAST if total == I31 else ("FFFHFF" if strand == "+" else ON)
        case("total-%d-two-nodes%s" % (total, strand), t, gaf("tot", 150, 10, 115, strand, ">o1>t", 50, 150, 95, 105, "50M5I50M"), rt)
        case("total-%d-interval-first%s" % (total, strand), t + "big\t1000\n", gaf("tot", 150, 10, 115, strand, "<big:0-100<t", 50, 150, 95, 105, "50M5I50M"), rt)
        case("total-%d-empty-step%s" % (total, strand), t + "zero\t0\n", gaf("tot", 150, 10, 115, strand, ">o1:0-100>zero:7-7>t", 50, 150, 95, 105, "50M5I50M"), rt)
        case("total-%d-intervals%s" % (total, strand), t, gaf("tot", 150, 10, 145, strand, ">o1:0-50<o1:50-100>t", 20, 150, 130, 135, "65M5I65M"), rt)


# CIGAR ops at the digit-count boundaries of the decoders: 3/4 digits (k_rec's and k_par's windows), 4/5 (k_fuse's SWAR
# window), 7/8 (every kernel), and 8-digit ops below and above 2^24 (k_par keeps 24 bits of an op).  Matches, and
# insertions / deletions between matches; and an op cut by a step boundary inside it.
for x in (999, 1000, 9999, 10000, 9999999, 10000000, 16777217, 99999999, 100000000):
    rt = FAST if x <= 9999999 else ("HHHHFF" if x <= 99999999 else ON)   # k_long reads ops of up to 8 digits
    for strand in "+-":
        case("op-%dM%s" % (x, strand), "big\t%d\n" % I31, gaf("op", x + 50, 10, x + 10, strand, ">big", 1000, 1000 + x, x, x, "%dM" % x), rt)
        case("op-%dI%s" % (x, strand), "big\t%d\n" % I31, gaf("op", x + 150, 10, x + 110, strand, ">big", 1000, 1100, 100, x + 100, "50M%dI50M" % x), rt)
        case("op-%dD%s" % (x, strand), "big\t%d\n" % I31, gaf("op", 150, 10, 110, strand, "<big", 1000, 1100 + x, 100, x + 100, "50M%dD50M" % x), rt)
        cut = x // 2 + 17
        case("op-%dM-cut%s" % (x, strand), "n1\t%d\nn2\t%d\n" % (cut, x),
             gaf("op", x + 50, 10, x + 10, strand, ">n1<n2", 0, x, x, x, "%dM" % x), rt)
        case("op-%dD-cut%s" % (x, strand), "n1\t%d\nn2\t%d\n" % (cut + 40, x + 100),
             gaf("op", 150, 10, 110, strand, ">n1>n2", 0, x + 100, 100, x + 100, "50M%dD50M" % x), rt)


# Query coordinates past 2^31 (k_par keeps the query coordinate as a u32 and the record's block sum in 31 bits; k_long
# keeps q0 + q, nm and nb of a line in 31 bits): long records of many 7-digit insertions.  Too long for k_fuse, k_rec
# and k_short.
def long_ins(qs, q, strand, m_col=200, path=">o1>o2", ps=50, pe=130):
    """qs and a query span q made of 50M + insertions + a target remainder (W = pe - ps)."""
    w = pe - ps
    ins = q - w
    n, r = divmod(ins, 9999999)
    cg = "%dM" % (w // 2) + "9999999I" * n + ("%dI" % r if r else "") + "%dM" % (w - w // 2)
    return gaf("ql", 999999999, qs, 999999999, strand, path, ps, pe, m_col, 999999999, cg)   # (qlen and qe: 9 digits)


QS = 999999999
for strand in "+-":
    case("q1-2^31-1" + strand, "", long_ins(QS, I31 - QS, strand), "HHHFFF")          # k_long's own limit: q1 <= 2^31-1
    case("q1-2^31" + strand, "", long_ins(QS, 2 ** 31 - QS, strand), "HHHFHH")
    case("q1-2^32" + strand, "", long_ins(QS, 2 ** 32 - QS, strand), ON)               # (its block sum is past 2^31-1)
    case("block-2^31-1" + strand, "", long_ins(QS, I31, strand), "HHHFHH")           # the largest q1 k_par takes: 3147483646
    case("block-2^31" + strand, "", long_ins(QS, 2 ** 31, strand), ON)
    case("nb-2^31-1" + strand, "", long_ins(0, I31, strand, path=">o1", ps=0, pe=80), "HHHFFF")   # nb of the one line
    case("nb-2^31" + strand, "", long_ins(0, 2 ** 31, strand, path=">o1", ps=0, pe=80), ON)
    case("nb-2^31-1-two-lines" + strand, "", long_ins(0, I31, strand), "HHHFFF")       # the insertions are in the first line
    # nm of a line: the window (pe - ps, 9 digits) bounds it below 10^9
    case("nm-999999999" + strand, "big\t%d\n" % I31,
         gaf("nm", 999999999, 0, 999999999, strand, ">big", 0, 999999999, 999999999, 999999999, "9999999M" * 100 + "99M"), "FHHFFF")   # 901 bytes: k_fuse takes it

# gi:f: (matches / block, rounded to 1/1000 in double): the 0..1 fast formatters, or handed on
for strand in "+-":
    def gi(m, b, name, rt):
        case("gi-%s%s" % (name, strand), "", gaf("gi", 150, 10, 115, strand, ">o1", 0, 100, m, b, "50M5I50M"), rt)
    gi(101, 100, "m-above-b", ON)
    gi(999999999, 1, "m-far-above-b", ON)
    gi(95, 0, "b-zero", FAST)
    gi(95, "*", "b-star", "HFFFFF")   # k_fuse copies matches and block verbatim: plain decimals only
    gi(95, -7, "b-negative", ON)
    gi("*", 2000, "m-star-rounds-to-0", "HFFFFF")
    gi("*", 100, "m-star", ON)
    gi(-5, 100, "m-negative", ON)
    gi(2 ** 53 + 1, 2 ** 53 + 3, "m-above-2^53", ON)
    gi(9007199254740993, 9007199254740993, "m-equals-b-above-2^53", ON)
    for k in (0, 1, 499, 500, 998, 999):
        gi(2 * k + 1, 2000, "tie-%d" % k, FAST)
        gi((2 * k + 1) * 499999, 2000 * 499999, "tie-9-digits-%d" % k, FAST)
    gi(999999999, 999999999, "one", FAST)
    gi(1, 999999999, "tiny", FAST)

@pytest.fixture(scope="module")
def td():
    with tempfile.TemporaryDirectory() as d:
        yield d


@pytest.mark.parametrize("name,lengths,records,routes", CASES, ids=[c[0] for c in CASES])
def test_limit_case(td, name, lengths, records, routes):
    bad = check_case(td, lengths, records, routes)
    assert not bad, "\n".join(bad)


# ---- a seeded generator of valid records with numbers of 1-10 digits ---------------------------------------------
def loguniform(rnd, lo, hi):
    return min(hi, int(math.exp(rnd.uniform(math.log(lo), math.log(hi + 1))))) if hi > lo else lo


def gen_batch(seed, n=2000):
    """-> (lengths TSV, GAF text): n valid records whose numbers are drawn log-uniformly over 1-10 digits, on nodes
    whose lengths cluster around 2^31 and 2^32 (and small ones); every CIGAR covers its path window exactly, so that
    the records convert (or are handed on) instead of aborting the reference."""
    rnd = random.Random(seed)
    nodes = {}
    for i in range(300):
        k = rnd.random()
        if k < 0.5:
            L = loguniform(rnd, 1, 10 ** 6)
        elif k < 0.7:
            L = loguniform(rnd, 10 ** 6, 10 ** 10)
        else:
            L = rnd.choice((2 ** 31, 2 ** 32)) + rnd.randrange(-3, 3) * rnd.choice((1, 1, 100, 10 ** 6))
        nodes["n%d" % i] = L
    small = [k for k, v in nodes.items() if v <= 10 ** 6]
    recs = []
    while len(recs) < n:
        nst = rnd.choice((1, 1, 1, 2, 2, 3))
        names = [rnd.choice(list(nodes)) for _ in range(nst)]
        names[1:-1] = [rnd.choice(small) for _ in names[1:-1]]
        steps, lens = [], []
        for nm in names:
            L = nodes[nm]
            if rnd.random() < 0.2 and L > 2:   # interval step
                a = rnd.randrange(0, min(L, 10 ** 10) - 1)
                b = a + loguniform(rnd, 1, min(L - a, 10 ** 9))
                steps.append("%s%s:%d-%d" % (rnd.choice("><"), nm, a, b))
                lens.append(b - a)
            else:
                steps.append(rnd.choice("><") + nm)
                lens.append(L)
        total = sum(lens)
        if nst == 1:
            ps = rnd.randrange(0, total) if rnd.random() < 0.3 else total - loguniform(rnd, 1, total)
            pe = ps + loguniform(rnd, 1, min(total - ps, 10 ** 9))
        else:   # the window starts in the first step and ends in the last
            ps = lens[0] - loguniform(rnd, 1, min(lens[0], 10 ** 6))
            pe = total - lens[-1] + loguniform(rnd, 1, min(lens[-1], 10 ** 6))
        w = pe - ps
        if w > 3 * 10 ** 9:
            continue
        ops, left, q = [], w, 0
        while left > 0:
            x = min(left, loguniform(rnd, 1, rnd.choice((10 ** 3, 10 ** 7, 10 ** 8))))
            if left > 30 * 10 ** 7 and x < left // 30:
                x = min(left, rnd.randrange(left // 30, left // 10 + 2))
            c = rnd.choice("MMMM=XD")
            ops.append("%d%s" % (x, c))
            left -= x
            q += 0 if c == "D" else x
            if rnd.random() < 0.3:
                y = loguniform(rnd, 1, rnd.choice((10, 10 ** 4, 10 ** 7, 10 ** 8)))
                ops.append("%dI" % y)
                q += y
        if ops[-1].endswith("I"):
            ops.pop()
        if not any(o.endswith(("M", "=")) for o in ops):
            ops[0] = ops[0][:-1] + "M"   # (the first op consumes target bases)
        if len(ops) > 400:
            continue
        num = lambda: loguniform(rnd, 1, 10 ** 10)
        qs = num() - 1
        b = num()
        m = rnd.choice((b, rnd.randrange(0, b + 1), num()))
        recs.append(gaf("g%d" % len(recs), num(), qs, num(), rnd.choice("+-"), "".join(steps), ps, pe, m, b, "".join(ops),
                        mapq=rnd.choice((0, 60, 254, 255, 1000)), plen=num(), tags=rnd.choice(((), ("tp:A:P",), ("tp:A:S", "rc:Z:a")))))
    lengths = "".join("%s\t%d\n" % kv for kv in nodes.items())
    return lengths, ("\n".join(recs) + "\n").encode()


def pad_all(data):
    return data.replace(b"\tcg:Z:", ("\t" + PAD + "\tcg:Z:").encode())


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_generated_batch(td, seed):
    """Every configuration on a seeded batch: the reference's bytes, and in each fast configuration both some records
    converted by its kernel and some handed on."""
    lengths, data = gen_batch(seed)
    lp = os.path.join(td, "g%d.tsv" % seed)
    with open(lp, "w") as f:
        f.write(lengths)
    nrec = data.count(b"\n")
    rc, ref, err = oracle(lp, data)
    assert rc == 0 and ref.count(b"\n") > nrec // 2, err[-300:]
    for cfg in ORDER:
        binary, env, pad = CONFIGS[cfg]
        d = pad_all(data) if pad else data
        if pad:
            rc, ref, err = oracle(lp, d)
            assert rc == 0
        grc, out, st = run_simt(binary, env, lp, d)
        assert grc == 0 and out == ref, cfg
        assert st[0] == "pipe", (cfg, st)   # k_fuse converts a batch whole or not at all: see test_generated_fuse
        _, n, to_par, steps, to_long, general = st
        if cfg in ("fuse", "rec", "short"):   # (fuse: the general pipeline's k_rec, after k_fuse handed the batch on)
            assert 0 < to_par < n, (cfg, st)
        elif cfg == "par":
            assert to_par == n and steps > 0 and 0 < to_long < n, (cfg, st)
        else:
            assert to_par == to_long == n and 0 < general < n, (cfg, st)


@pytest.mark.parametrize("seed", [1])
def test_generated_fuse(td, seed):
    """k_fuse takes a batch whole or hands it on whole: the records k_rec converts of a generated batch (those of at
    most 240 bytes that the general kernel did not print) go through k_fuse in one batch, the others in another."""
    lengths, data = gen_batch(seed, n=200)
    lp = os.path.join(td, "f%d.tsv" % seed)
    with open(lp, "w") as f:
        f.write(lengths)
    recs = data.split(b"\n")[:-1]
    fast, rest = [], []
    for r in recs:   # one record at a time through k_rec: converted or handed on
        _, _, st = run_simt(SIMT, {"G2P_FUSE": "0"}, lp, r + b"\n")
        (fast if st[2] == 0 else rest).append(r)
    assert len(fast) > 20 and len(rest) > 20
    for part, want in ((fast, True), (rest, False)):
        d = b"\n".join(part) + b"\n"
        rc, ref, err = oracle(lp, d)
        grc, out, st = run_simt(SIMT, {"G2P_FUSE": "2"}, lp, d)
        assert rc == grc == 0 and out == ref
        assert (st == ("fused", len(part))) == want, st


# ---- the same on the GPU ------------------------------------------------------------------------------------------
GPU_CONFIGS = ("fuse", "rec", "short", "par", "long")   # (g2p_simt_long's kernels are a build of the emulator only)


def gpu_route(cfg, res, nrec, k):
    """As route_of, from the counters of struct g2p_result."""
    fused, to_par, par, general = res.n_fused, res.n_long, res.n_par, res.n_delegated
    if cfg == "fuse":
        return "F" if fused == nrec else ("H" if fused == 0 else "fused %d" % fused)
    got = (fused, to_par, par, general)
    if fused:
        return repr(got)
    if cfg in ("rec", "short"):
        return {0: "F", k: "H"}.get(to_par, repr(got))
    if to_par != k:
        return repr(got)
    if cfg == "par":
        return {k: "F", 0: "H"}.get(par, repr(got))
    return {0: "F", k: "H"}.get(general, repr(got)) if par == 0 else repr(got)


@pytest.fixture(params=GPU_CONFIGS)
def gpu_cfg(request, g2p, monkeypatch):
    """(configuration, Converter created under its environment: g2p_create reads the variables)."""
    for k, v in CONFIGS[request.param][1].items():
        monkeypatch.setenv(k, v)
    cv = g2p.Converter(0)
    yield request.param, cv
    cv.close()


@pytest.mark.gpu
def test_gpu_limit_cases(g2p, gpu_cfg, td):
    cfg, cv = gpu_cfg
    _, _, pad = CONFIGS[cfg]
    lp = os.path.join(td, "gpu.tsv")
    bad = []
    for name, lengths, records, routes in CASES:
        with open(lp, "w") as f:
            f.write(BASE_LENGTHS + lengths)
        data = batch(records, pad)
        rc, ref, err = oracle(lp, data)
        assert rc == 0, name
        assert cv.load_lengths((BASE_LENGTHS + lengths).encode())
        out, res = cv.convert_host(data)
        if g2p.exit_code(res) != 0 or out != ref:
            bad.append("%s: bytes differ from the reference" % name)
            continue
        got = gpu_route(cfg, res, data.count(b"\n"), len(records))
        if got != dict(zip(ORDER, routes))[cfg]:
            bad.append("%s: route %s, want %s" % (name, got, dict(zip(ORDER, routes))[cfg]))
    assert not bad, "\n".join(bad[:40])


@pytest.mark.gpu
def test_gpu_generated_batches(g2p, gpu_cfg, td):
    cfg, cv = gpu_cfg
    for seed in (1, 2):
        lengths, data = gen_batch(seed)
        if CONFIGS[cfg][2]:
            data = pad_all(data)
        lp = os.path.join(td, "gg.tsv")
        with open(lp, "w") as f:
            f.write(lengths)
        rc, ref, err = oracle(lp, data)
        assert rc == 0
        assert cv.load_lengths(lengths.encode())
        out, res = cv.convert_host(data)
        assert g2p.exit_code(res) == 0 and out == ref, (cfg, seed)
        n = data.count(b"\n")
        assert res.n_fused == 0, (cfg, seed)   # k_fuse hands a batch with any record it cannot take on whole
        if cfg in ("fuse", "rec", "short"):
            assert 0 < res.n_long < n, (cfg, seed)
        elif cfg == "par":
            assert res.n_long == n and 0 < res.n_par < n, (cfg, seed)
        else:
            assert res.n_long == n and res.n_par == 0 and 0 < res.n_delegated < n, (cfg, seed)


def combined(prefixes=None):
    """Every case record (or those of the cases whose names start with one of `prefixes`), unpadded, between ordinary
    records in one file, the case's own nodes renamed per case."""
    lengths, recs = [BASE_LENGTHS], []
    for i, (name, ln, records, routes) in enumerate(CASES):
        if prefixes and not name.startswith(prefixes):
            continue
        names = [l.split("\t")[0] for l in ln.splitlines()]
        ren = lambda nm: "c%d%s" % (i, nm) if nm in names else nm
        lengths += ["%s\t%s\n" % (ren(l.split("\t")[0]), l.split("\t")[1]) for l in ln.splitlines()]
        for r in records:
            c = r.split("\t")
            c[5] = re.sub(r"([<>])([^<>:]+)", lambda m: m.group(1) + ren(m.group(2)), c[5])
            recs += ["\t".join(c), ORDINARY[i % 4]]
    return "".join(lengths), ("\n".join(recs) + "\n").encode()


@pytest.mark.gpu
def test_gpu_combined_cli_and_device_filter(g2p, td):
    """All cases in one file through the gaf2paf executable; then the same batch through g2p_convert_device into
    g2p_filter_device, whose PAF has query starts above 2^31 for the filter to compare."""
    import torch
    lengths, data = combined()
    lp, gp = os.path.join(td, "all.tsv"), os.path.join(td, "all.gaf")
    with open(lp, "w") as f:
        f.write(lengths)
    with open(gp, "wb") as f:
        f.write(data)
    rc, ref, err = oracle(lp, data)
    assert rc == 0
    assert max(int(l.split(b"\t")[2]) for l in ref.splitlines()) > 2 ** 31
    crc, cout, cerr = H.run_tool(EXE, [gp, "-l", lp])
    assert crc == 0 and cout == ref, cerr[-300:]
    # the device-resident path on the records whose query coordinates pass 2^31 (several alignments per query name)
    lengths, data = combined(("q1-", "block-", "nb-"))
    with open(lp, "w") as f:
        f.write(lengths)
    rc, ref, err = oracle(lp, data)
    assert rc == 0 and max(int(l.split(b"\t")[2]) for l in ref.splitlines()) > 2 ** 31
    fbin, _ = H.oracle_path("auto", "gaffilter")
    frc, fref, ferr = H.run_tool(fbin, ["-r", "2", "-p", "-"], ref)
    assert frc == 0 and 0 < fref.count(b"\n") < ref.count(b"\n"), ferr[-300:]
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths.encode())
        t = torch.empty(len(data) + 16, dtype=torch.uint8, device="cuda")
        g2p.copy_to_device(t.data_ptr(), data)
        torch.cuda.synchronize()
        stream = torch.cuda.current_stream().cuda_stream
        d_paf, r1 = cv.convert_device(t.data_ptr(), len(data), stream)
        assert g2p.exit_code(r1) == 0 and r1.out_bytes == len(ref)
        assert g2p.copy_to_host(d_paf, r1.out_bytes) == ref
        d_out, r2 = cv.filter_device(d_paf, r1.out_bytes, g2p.Converter.filter_params(ratio=2.0, paf=True), stream)
        assert g2p.exit_code(r2) == 0
        assert g2p.copy_to_host(d_out, r2.out_bytes) == fref
    finally:
        cv.close()


def test_combined_file_under_the_emulator(td):
    """The combined file of the GPU test, under the emulator: renaming the nodes keeps every case valid."""
    lengths, data = combined()
    lp = os.path.join(td, "all.tsv")
    with open(lp, "w") as f:
        f.write(lengths)
    rc, ref, err = oracle(lp, data)
    assert rc == 0, err[-300:]
    grc, out, st = run_simt(SIMT, {"G2P_FUSE": "0"}, lp, data)
    assert grc == 0 and out == ref and 0 < st[2] < st[1]
