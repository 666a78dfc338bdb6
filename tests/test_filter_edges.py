"""gaffilter at the places where its kernels (csrc/g2p_filter.cuh) could be subtly wrong, compared with the reference
gaffilter or, without the reference build, its independent restatement oracle/bin/gaffilter_oracle (see test_filter.py):

* the sort and the segmented max-scan: colliding 32-bit name hashes, names of 16 / 17 bytes, runs that start and end at
  the 2048-entry tiles, a long interval carried across tiles, singletons, duplicates, '*' lines inside a run;
* interval geometry: touching and nested intervals, empty records, negative starts, the largest sortable start;
* the double arithmetic at option thresholds (-r, -m, -o, -b, -q, -i), rc / tp tags, PAF gl / gm;
* the float parse of gi tags (std::stof: correctly rounded, out-of-range values throw);
* a seeded mutation fuzz.

CPU tests run the kernels under the SIMT emulator (build/g2p_filter_simt); the GPU tests (-m gpu) run the same files
through the C-ABI, the gaffilter executable and the device-resident gaf2paf -> filter path.  Every differential case
filters some records and keeps others."""
import os
import random
import struct
import subprocess
import time

import pytest

import helpers as H
from test_filter import assert_partial, last_line, ref_gaffilter, simt

FLOATPARSE = os.path.join(H.BUILD, "g2p_floatparse")
K_TILE = 2048   # kRsTile == kSegTile


def gaf(name, qs, qe, mapq=60, block=None, matches=None, qlen=None, tags=(), path=">a"):
    block = max(qe - qs, 0) if block is None else block
    matches = block if matches is None else matches
    qlen = max(qs, qe) + 10 if qlen is None else qlen
    cols = [name, qlen, qs, qe, "+", path, 1000000, 0, max(block, 1), matches, block, mapq] + list(tags)
    return ("\t".join(str(c) for c in cols) + "\n").encode()


def paf(name, qs, qe, mapq=60, block=None, matches=None, qlen=None, tags=()):
    block = max(qe - qs, 0) if block is None else block
    matches = block if matches is None else matches
    qlen = max(qs, qe) + 10 if qlen is None else qlen
    cols = [name, qlen, qs, qe, "+", "t1", 1000000, 0, max(block, 1), matches, block, mapq] + list(tags or ["cg:Z:%dM" % max(block, 1)])
    return ("\t".join(str(c) for c in cols) + "\n").encode()


def f32(x):
    return struct.unpack("<f", struct.pack("<f", x))[0]


def f32_next(x, up):
    b = struct.unpack("<I", struct.pack("<f", x))[0]
    return struct.unpack("<f", struct.pack("<I", b + (1 if up else -1)))[0]


# ---- the sort key and the segmented scan ---------------------------------------------------------------------------
def collision_case(names, rnd, line=gaf):
    """Names whose 32-bit sort hashes collide, their records interleaved in one sorted run.  Every other name holds a
    strong record and a weak one it filters; the names between hold one weak record alone on its query, which is kept --
    and would be filtered if the kernels took the colliding names for one query."""
    out = []
    for k, nm in enumerate(names):
        s = 3 * k
        if k % 2 == 0:
            out += [line(nm, s, s + 100, mapq=60), line(nm, s + 50, s + 150, mapq=5)]
        else:
            out += [line(nm, s + 1, s + 101, mapq=1)]
    rnd.shuffle(out)
    return b"".join(out)


def run_case(n, rnd, long_first=False, line=gaf, name="contig_1", step=10):
    """One query sequence with `n` records spread along it (a run of n sorted entries).  long_first: record 0 covers the
    whole run with the highest MAPQ -- every later record, in every tile of the scan, has to find it through the carried
    running maximum."""
    out = []
    for k in range(n):
        s = step * k + rnd.randrange(10)
        ln = rnd.choice([5, 20, 60, 200]) if rnd.random() < 0.97 else 3000
        out.append(line(name, s, s + ln, mapq=rnd.choice([0, 1, 5, 20, 60, 60, 60]),
                        tags=["tp:A:%s" % rnd.choice("PPPS")] if line is gaf else ["tp:A:%s" % rnd.choice("PPPS"), "cg:Z:%dM" % ln]))
    if long_first:
        out = [line(name, 0, step * n + 500, mapq=60, block=40 * n)] + out
    rnd.shuffle(out)
    return b"".join(out)


def sort_scan_cases():
    rnd = random.Random(5)
    w = ["aaaa", "bbbb", "cccc", "dddd"]
    names8 = ["aaaabbbb", "bbbbaaaa", "ccccdddd", "ddddcccc"]
    names16 = [a + b + c + d for a in w for b in w for c in w for d in w if len({a, b, c, d}) == 4][:12]
    names1617 = ["abcdefghijklmnop", "abcdefghijklmnopq", "abcdefghijklmnopr", "bbcdefghijklmnop", "abcdefghijklmnopqrstuvwxyz0123456"]
    cases = [
        ("hash32_8", collision_case(names8, rnd), ["-r", "2"]),
        ("hash32_16", collision_case(names16, rnd), ["-r", "2"]),
        ("hash32_16_paf", collision_case(names16, rnd, paf), ["-r", "2", "-p"]),
        ("names_16_17", collision_case(names1617, rnd), ["-r", "2"]),
    ]
    for n in (K_TILE - 1, K_TILE, K_TILE + 1, 3 * K_TILE + 5):
        # the run surrounded by other records: it starts inside a tile and ends at / across its boundaries
        text = run_case(n, rnd) + gaf("a_before", 0, 100, mapq=60) + gaf("a_before", 10, 90, mapq=1) + gaf("zz_after", 0, 50)
        cases.append(("run_%d" % n, text, ["-r", "2"]))
        cases.append(("run_%d_exact" % n, run_case(n, rnd, step=40), ["-r", "2"]))
    cases.append(("carry_across_tiles", run_case(3 * K_TILE + 700, rnd, long_first=True), ["-r", "2"]))
    cases.append(("carry_across_tiles_paf", run_case(3 * K_TILE + 700, rnd, long_first=True, line=paf), ["-r", "2", "-p"]))
    single = [gaf("s%d" % k, k % 50, k % 50 + 30, mapq=rnd.choice([1, 60])) for k in range(3000)]
    single += [gaf("s%d" % k, 5, 25, mapq=1) for k in range(0, 3000, 7)]
    rnd.shuffle(single)
    cases.append(("singletons", b"".join(single), ["-r", "2"]))
    dup = gaf("d1", 0, 50, mapq=60, tags=["tp:A:P", "rc:Z:x"])
    cases.append(("duplicates", dup * 3 + gaf("d1", 60, 90) + gaf("d2", 0, 50) + dup, ["-r", "1"]))
    cases.append(("duplicates_o", dup * 2 + gaf("d2", 0, 500, block=500) + gaf("d2", 5, 50, block=30), ["-o", "40"]))
    star = b"*\t>s43\t97\t12\t0\t6\t92\n"
    text = b"".join(gaf("st", 10 * k, 10 * k + 15, mapq=[60, 1][k % 2]) + (star if k % 3 == 0 else b"") for k in range(40))
    cases.append(("star_lines_in_run", star + text + star, ["-r", "2"]))
    return cases


# ---- interval geometry ---------------------------------------------------------------------------------------------
def geometry_cases():
    keep = gaf("other", 0, 10) + gaf("other2", 0, 10, mapq=1) + gaf("other2", 2, 8, mapq=60)
    return [
        # [0, 50) and [50, 100): closed intervals [0, 49] and [50, 99] do not overlap; [0, 51) reaches 50
        ("touching", gaf("t1", 0, 50, mapq=60) + gaf("t1", 50, 100, mapq=1) + gaf("t2", 0, 51, mapq=60) + gaf("t2", 50, 100, mapq=1), ["-r", "2"]),
        ("touching_o", gaf("t1", 0, 50) + gaf("t1", 50, 100) + gaf("t2", 0, 51) + gaf("t2", 50, 100, block=10), ["-o", "20"]),
        ("nested_equal_starts", gaf("n", 0, 100, mapq=60) + gaf("n", 0, 50, mapq=20) + gaf("n", 10, 20, mapq=60) + gaf("n", 0, 100, mapq=1, tags=["tp:A:S"])
         + gaf("n", 100, 200, mapq=5) + gaf("m", 5, 6) + gaf("m", 5, 7, mapq=30), ["-r", "2"]),
        ("empty_alone", gaf("e1", 10, 10, mapq=60) + gaf("e2", 10, 10) + gaf("e2", 0, 40, mapq=1) + gaf("e3", 0, 0) + keep, ["-r", "2"]),
        ("empty_inside", gaf("e1", 20, 20, mapq=60) + gaf("e1", 0, 40, mapq=1) + gaf("e1", 5, 30, mapq=60) + keep, ["-o", "10"]),
        # two empty records next to each other: [9, 10] meets [10, 10]... overlap_size's assert(oend >= ostart) fires
        ("empty_neighbours", gaf("e", 10, 10) + gaf("e", 11, 11) + keep, ["-r", "2"]),
        ("negative_starts", gaf("ng", -20, 30, mapq=60) + gaf("ng", -5, -1, mapq=1) + gaf("ng", -30, -25, mapq=1) + gaf("ng", 0, 10, mapq=5) + keep, ["-r", "2"]),
        ("largest_start", gaf("big", 4294967280, 4294967380, mapq=60) + gaf("big", 4294967200, 4294967290, mapq=1)
         + gaf("big", 4294967000, 4294967100, mapq=1) + keep, ["-r", "2"]),
    ]


# ---- thresholds ------------------------------------------------------------------------------------------------------
def threshold_cases():
    # a / (b + 0.000001) == ratio exactly in double for b = 0: 2 / 0.000001 == 2000000, 3 / 0.000001 == 3000000
    assert 2 / (0 + 0.000001) == f32(2000000) and 3 / (0 + 0.000001) == f32(3000000)
    fi = f32(0.95)
    below, above = f32_next(fi, False), f32_next(fi, True)
    ident = lambda g: ["gi:f:%.9g" % g]
    cases = [
        # dominates(): g1.mapq / (g2.mapq + 1e-6) >= ratio (kept), g2.mapq / (g1.mapq + 1e-6) >= ratio (filtered although
        # its block is longer), g1.block / (g2.block + 1e-6) >= ratio
        ("ratio_tie_mapq", gaf("a", 0, 50, mapq=2, block=1) + gaf("a", 10, 60, mapq=0, block=0) + gaf("b", 0, 50, mapq=0, block=5) + gaf("b", 10, 60, mapq=2, block=0),
         ["-r", "2000000"]),
        ("ratio_tie_block", gaf("a", 0, 50, mapq=0, block=3) + gaf("a", 10, 60, mapq=0, block=0) + gaf("b", 0, 50, mapq=0, block=2) + gaf("b", 10, 60, mapq=0, block=0),
         ["-r", "3000000"]),
        ("ratio_mapq_60_30", gaf("a", 0, 50, mapq=60) + gaf("a", 10, 60, mapq=30) + gaf("b", 0, 50, mapq=60) + gaf("b", 10, 60, mapq=29)
         + gaf("c", 0, 50, mapq=255) + gaf("c", 10, 60, mapq=0) + gaf("d", 0, 50, mapq=0) + gaf("d", 10, 60, mapq=0, block=20), ["-r", "2"]),
        ("ratio_1", gaf("a", 0, 50) + gaf("a", 10, 60) + gaf("b", 0, 50, mapq=61) + gaf("b", 10, 60) + gaf("c", 0, 50, block=51) + gaf("c", 10, 60), ["-r", "1"]),
        # -m: overlap / block_length >= float(option); 0.25 is exact, 0.1 is not
        ("min_overlap_eq", gaf("a", 0, 100, mapq=1) + gaf("a", 75, 200, mapq=60) + gaf("b", 0, 100, mapq=1) + gaf("b", 76, 200, mapq=60), ["-r", "2", "-m", "0.25"]),
        # float(0.1) == 13421773 / 2^27: an overlap of 13421773 over a block of 2^27 is just enough, 10 / 100 is not
        ("min_overlap_float", gaf("a", 0, 100, mapq=1) + gaf("a", 90, 200, mapq=60) + gaf("b", 0, 100, mapq=1) + gaf("b", 89, 200, mapq=60)
         + gaf("c", 0, 2 ** 27, mapq=1) + gaf("c", 2 ** 27 - 13421773, 2 ** 28, mapq=60) + gaf("d", 0, 2 ** 27, mapq=1) + gaf("d", 2 ** 27 - 13421772, 2 ** 28, mapq=60),
         ["-r", "2", "-m", "0.1"]),
        ("min_overlap_len_eq", gaf("a", 0, 100, block=100) + gaf("a", 50, 150, block=99) + gaf("b", 0, 100, block=101) + gaf("b", 50, 150, block=100), ["-o", "100"]),
        ("min_block_eq", gaf("a", 0, 100, mapq=1) + gaf("a", 10, 60, mapq=60, block=50, qlen=500) + gaf("b", 0, 100, mapq=1) + gaf("b", 10, 60, mapq=60, block=49, qlen=500)
         + gaf("c", 0, 100, mapq=1) + gaf("c", 10, 60, mapq=60, block=49, qlen=50) + gaf("d", 0, 100, mapq=1) + gaf("d", 10, 60, mapq=60, block=49, qlen=51),
         ["-r", "2", "-b", "50"]),
        ("min_mapq_eq", gaf("a", 0, 100, mapq=1) + gaf("a", 10, 60, mapq=5) + gaf("b", 0, 100, mapq=1) + gaf("b", 10, 60, mapq=4), ["-r", "2", "-q", "5"]),
        # -i against gi one float ulp either side of float(0.95) (identity = min(block / matches, gi))
        ("min_identity_ulp", gaf("a", 0, 100, mapq=1) + gaf("a", 10, 60, mapq=60, tags=ident(fi)) + gaf("b", 0, 100, mapq=1) + gaf("b", 10, 60, mapq=60, tags=ident(below))
         + gaf("c", 0, 100, mapq=1) + gaf("c", 10, 60, mapq=60, tags=ident(above)) + gaf("d", 0, 100, mapq=1) + gaf("d", 10, 60, mapq=60, block=19, matches=20),
         ["-r", "2", "-i", "0.95"]),
        ("rc_tags", gaf("a", 0, 100, mapq=1, tags=["rc:Z:chr1"]) + gaf("a", 10, 60, mapq=60, tags=["rc:Z:chr1"]) + gaf("b", 0, 100, mapq=1, tags=["rc:Z:chr1"])
         + gaf("b", 10, 60, mapq=60, tags=["rc:Z:chr2"]) + gaf("c", 0, 100, mapq=1) + gaf("c", 10, 60, mapq=60, tags=["rc:Z:chr2"])
         + gaf("d", 0, 100, mapq=1, tags=["rc:Z:chr1"]) + gaf("d", 10, 60, mapq=60), ["-r", "2"]),
        ("tp_tags", gaf("a", 0, 100, mapq=1, tags=["tp:A:P"]) + gaf("a", 10, 60, mapq=60, tags=["tp:A:S"]) + gaf("b", 0, 100, mapq=1) + gaf("b", 10, 60, mapq=60, tags=["tp:A:S"])
         + gaf("c", 0, 100, mapq=1, tags=["tp:A:I"]) + gaf("c", 10, 60, mapq=60, tags=["tp:A:S"]) + gaf("d", 0, 100, mapq=1, tags=["tp:A:PP"]) + gaf("d", 10, 60, mapq=60),
         ["-r", "2"]),
        ("paf_tp_gl_gm", paf("a", 0, 100, mapq=1, tags=["tp:A:S", "tp:A:P", "cg:Z:100M"]) + paf("a", 10, 60, mapq=60, tags=["tp:A:P", "tp:A:S", "cg:Z:50M"])
         + paf("b", 0, 100, mapq=60, block=10, tags=["gl:i:300", "cg:Z:100M"]) + paf("b", 10, 60, mapq=60, tags=["cg:Z:50M"])
         + paf("c", 0, 100, mapq=60, tags=["gm:i:0", "gl:i:5", "cg:Z:100M"]) + paf("c", 10, 60, mapq=60, block=200)
         + paf("d", 0, 100, mapq=1, tags=["rc:Z:x", "cg:Z:100M"]) + paf("d", 10, 60, mapq=60, tags=["rc:Z:y", "cg:Z:50M"]), ["-r", "2", "-p"]),
        ("paf_gl_identity", paf("a", 0, 100, mapq=1) + paf("a", 10, 60, mapq=60, matches=50, tags=["gl:i:40", "cg:Z:50M"]) + paf("b", 0, 100, mapq=1)
         + paf("b", 10, 60, mapq=60, block=50, tags=["gm:i:60", "cg:Z:50M"]) + paf("c", 0, 100, mapq=1)
         + paf("c", 10, 60, mapq=60, matches=50, tags=["gl:i:60", "cg:Z:50M"]), ["-r", "2", "-i", "0.9", "-p"]),
        ("paf_block_o", paf("a", 0, 100, tags=["gl:i:150", "cg:Z:100M"]) + paf("a", 10, 60) + paf("b", 0, 100) + paf("b", 10, 60, tags=["gl:i:10", "cg:Z:50M"]), ["-o", "100", "-p"]),
    ]
    return cases


ALL_CASES = sort_scan_cases() + geometry_cases() + threshold_cases()
ABORTS = {"empty_neighbours"}


@pytest.mark.parametrize("name", [c[0] for c in ALL_CASES])
def test_emulated_filter_edges(name):
    text, args = next((t, a) for n, t, a in ALL_CASES if n == name)
    rc, out, err = ref_gaffilter(text, args)
    src, sout, serr = simt(text, args)
    assert src == rc == (134 if name in ABORTS else 0), (name, src, rc, serr[-300:], err[-300:])
    if rc == 0:
        assert sout == out
        assert last_line(serr) == last_line(err)
        assert_partial(err, name)
    else:
        assert sout == out == b""


def test_emulated_filter_unsupported_start():
    """A query start of 2^32 - 15 does not fit the sort key: reported, not mis-sorted (the emulator exits 98; the C-ABI
    returns an error, see test_gpu_filter_edges)."""
    text = gaf("big", 4294967281, 4294967380) + gaf("big", 4294967200, 4294967290, mapq=1)
    src, sout, serr = simt(text, ["-r", "2"])
    assert src == 98 and sout == b"" and "unsupported" in serr


# ---- gi: the float parse ---------------------------------------------------------------------------------------------
GI_EDGES = ["3.4028235e38", "3.4028234e38", "3.4028236e38", "1.2e-38", "1.17549435e-38", "1.17549432e-38", "1.1754943e-38", "1e-38",
            "1e-40", "1e-46", "1e40", "1e999", "3.5e38", "-1e-40", "-3.5e38", "0", "-0", "0.0e999", "0e-999", "1e-0001",
            "3.885933e+07", "1.361448e+09", "16777217", "16777219", "0.000000000000000000000000000000000000000000000123e44",
            "123456789012345678901234567890", "0.1000000000000000000000000000000000000001"]
# more than 19 significant digits within 10^-18 of a midpoint between two floats: not decided by the 19 digits kept, so
# rejected (a parse failure: the record aborts); stof rounds them (DESIGN §7)
GI_UNDECIDED = ["1.000000059604644775390625", "1.0000000596046447753906249999", "1.00000005960464477539062500000001"]


def floatparse(values):
    out = subprocess.run([FLOATPARSE], input=("\n".join(values) + "\n").encode(), stdout=subprocess.PIPE, check=True).stdout.decode()
    rows = [l.split() for l in out.strip().split("\n")]
    assert len(rows) == len(values)
    return rows


def gi_values():
    rnd = random.Random(7)
    vals = ["%g" % (k / 1e6) for k in range(1000001)]   # every %g value in [0, 1] at 6 significant digits
    for _ in range(100000):
        nd = rnd.randrange(7, 18)
        d = "".join(rnd.choice("0123456789") for _ in range(nd))
        p = rnd.randrange(nd + 1)
        vals.append(d[:p] + "." + d[p:])
    vals += ["%.6e" % (10 ** rnd.uniform(-20, 20)) for _ in range(100000)]
    vals += ["%.6e" % (10 ** rnd.uniform(5, 20)) for _ in range(50000)]
    return vals


def test_gi_parse_matches_stof():
    """parse_float_text (the kernels' std::stof of gi:f: values) is correctly rounded and rejects what stof rejects as
    out of range, on plain decimals: every %g value in [0, 1], 7-17-digit decimals, %.6e values from 1e-20 to 1e20 and the
    edges of the float range."""
    vals = gi_values() + GI_EDGES
    bad = [(v, r) for v, r in zip(vals, floatparse(vals)) if r[0] != r[1]]
    assert not bad, bad[:20]
    assert [r[0] for r in floatparse(GI_UNDECIDED)] == ["throw"] * len(GI_UNDECIDED)


def test_gi_out_of_range_aborts():
    """A gi value std::stof throws on ends the reference (uncaught std::out_of_range): exit 134, nothing printed."""
    base = gaf("a", 0, 100, mapq=1) + gaf("a", 10, 60, mapq=60) + gaf("b", 0, 10)
    for v in ("1e-40", "1e-38", "3.5e38", "1e40", "-1e-46"):
        text = base + gaf("c", 0, 50, tags=["gi:f:" + v])
        for args in (["-r", "2"], ["-r", "2", "-i", "0.5"]):
            rc, out, err = ref_gaffilter(text, args)
            src, sout, serr = simt(text, args)
            assert rc == src == 134 and out == sout == b"", (v, args)


def test_gi_rounding_decides_identity():
    """gi values whose correct rounding differs from a naive parse decide an -i threshold the way std::stof does."""
    # stof("3.885933e+07") == 38859328 (a tie, to even): below -i 38859332, so the gi record does not count
    cases = [("3.885933e+07", "38859332"), ("1.361448e+09", "1.36144806e9"), ("3.885933e+07", "38859328")]
    for gi, thr in cases:
        text = (gaf("q", 0, 100, mapq=1, block=40000000, matches=1) + gaf("q", 10, 60, mapq=60, block=1800000000, matches=1, tags=["gi:f:" + gi])
                + gaf("p", 0, 100, mapq=1) + gaf("p", 10, 60, mapq=60, block=2000000000, matches=1))
        rc, out, err = ref_gaffilter(text, ["-r", "2", "-i", thr])
        src, sout, serr = simt(text, ["-r", "2", "-i", thr])
        assert rc == src == 0 and sout == out and last_line(serr) == last_line(err), (gi, thr)
        assert_partial(err, (gi, thr))


# ---- seeded mutation fuzz (tests/fuzz_filter_vs_ref.py's mutations) ---------------------------------------------------
def paf_empty_tag_part(text):
    """PAF mode: an optional field with an empty ':'-separated part (the kernels print it as written: DESIGN §7)."""
    for line in text.split(b"\n"):
        for f in [x for x in line.split(b"\t") if x][12:]:
            if f.startswith(b":") or f.endswith(b":") or b"::" in f:
                return True
    return False


def test_emulated_filter_mini_fuzz():
    from fuzz_filter_vs_ref import OPTS
    from fuzz_vs_ref import mutate
    rnd = random.Random(11)
    partial = 0
    n = 300
    for it in range(n):
        paf_mode = rnd.random() < 0.5
        text, _ = H.gen_filter_case(700000 + it, n_records=40, n_queries=rnd.choice([3, 8, 12]), paf=paf_mode)
        lines = [l.decode("latin-1") for l in text.split(b"\n") if l]
        for _ in range(rnd.randrange(0, 3)):
            k = rnd.randrange(len(lines))
            lines[k] = mutate(rnd, lines[k].replace(" ", "\x01").replace("\t", " ")).replace("\x01", " ")
        data = ("\n".join(lines) + "\n").encode("latin-1")
        args = rnd.choice(OPTS) + (["-p"] if paf_mode else [])
        if paf_mode and paf_empty_tag_part(data):
            continue
        rc, out, err = ref_gaffilter(data, args)
        src, sout, serr = simt(data, args)
        assert src == rc and sout == out, (it, args, data)
        if rc == 0:
            assert last_line(serr) == last_line(err), (it, args)
            f, l = [int(x) for x in last_line(err).split("filtered ")[1].split(".")[0].split(" / ")]
            partial += 0 < f < l
    assert partial > n // 2


# ---- GPU -------------------------------------------------------------------------------------------------------------
def kwargs_of(args):
    names = {"-r": "ratio", "-m": "min_overlap", "-i": "min_identity", "-o": "min_overlap_length", "-b": "min_block_length", "-q": "min_mapq"}
    kw, i = {}, 0
    while i < len(args):
        if args[i] == "-p":
            kw["paf"] = True
            i += 1
        else:
            v = args[i + 1]
            kw[names[args[i]]] = float(v) if args[i] in ("-r", "-m", "-i") else int(v)
            i += 2
    return kw


def gpu_check(g2p, cv, exe, text, args, want_rc=0):
    rc, out, err = ref_gaffilter(text, args)
    assert rc == want_rc, (args, err[-200:])
    res_out, res = cv.filter_host(text, g2p.Converter.filter_params(**kwargs_of(args)))
    assert g2p.exit_code(res) == rc, args
    crc, cout, cerr = H.run_tool(exe, args + ["-"], text)
    assert crc == rc and cout == out, args
    if rc == 0:
        assert res_out == out, args
        assert "[gaffilter]: filtered %d / %d. total block lengths filtered: %d" % (res.n_filtered, res.n_loaded, res.filtered_len) == last_line(err)
        assert last_line(cerr) == last_line(err)
        assert_partial(err, args)
    return err


@pytest.mark.gpu
def test_gpu_filter_edges(g2p):
    """Every edge file of the emulator tests, and the gi cases, through Converter.filter_host and bin/gaffilter."""
    exe = os.path.join(g2p.BIN_DIR, "gaffilter")
    cv = g2p.Converter(0)
    try:
        for name, text, args in ALL_CASES:
            gpu_check(g2p, cv, exe, text, args, 134 if name in ABORTS else 0)
        base = gaf("a", 0, 100, mapq=1) + gaf("a", 10, 60, mapq=60) + gaf("b", 0, 10)
        gpu_check(g2p, cv, exe, base + gaf("c", 0, 50, tags=["gi:f:1e-40"]), ["-r", "2"], 134)
        for gi, thr in (("3.885933e+07", "38859332"), ("1.361448e+09", "1.36144806e9")):
            text = (gaf("q", 0, 100, mapq=1, block=40000000, matches=1) + gaf("q", 10, 60, mapq=60, block=1800000000, matches=1, tags=["gi:f:" + gi])
                    + gaf("p", 0, 100, mapq=1) + gaf("p", 10, 60, mapq=60, block=2000000000, matches=1))
            gpu_check(g2p, cv, exe, text, ["-r", "2", "-i", thr])
        # a start of 2^32 - 15 is refused by the device sort
        with pytest.raises(g2p.G2PError, match="query_start"):
            cv.filter_host(gaf("big", 4294967281, 4294967380) + gaf("big", 4294967200, 4294967290, mapq=1), g2p.Converter.filter_params(ratio=2))
    finally:
        cv.close()


@pytest.mark.gpu
def test_gpu_filter_device_resident_and_large(g2p):
    """gaf2paf -> filter_device with the PAF never leaving the device, on records spread along few long queries; then one
    large run (assembly contigs: a few queries with 10^5 alignments each among ~1.5 M records) through filter_host."""
    import torch
    cv = g2p.Converter(0)
    try:
        gaf_text = H.gen_spread_filter_case(91, n_records=40000, n_queries=4)
        _, lengths = H.gen_filter_case(91, n_records=10, n_queries=1)
        rc, paf_text, err, kind = H.run_gaf2paf_cpu(gaf_text, lengths)
        assert rc == 0
        assert cv.load_lengths(lengths)
        t = torch.empty(len(gaf_text) + 16, dtype=torch.uint8, device="cuda")
        g2p.copy_to_device(t.data_ptr(), gaf_text)
        torch.cuda.synchronize()
        stream = torch.cuda.current_stream().cuda_stream
        d_paf, r1 = cv.convert_device(t.data_ptr(), len(gaf_text), stream)
        assert g2p.exit_code(r1) == 0
        for args in (["-r", "2", "-p"], ["-o", "150", "-m", "0.2", "-p"]):
            rrc, rout, rerr = ref_gaffilter(paf_text, args)
            d_out, r2 = cv.filter_device(d_paf, r1.out_bytes, g2p.Converter.filter_params(**kwargs_of(args)), stream)
            assert rrc == 0 and g2p.exit_code(r2) == 0
            assert g2p.copy_to_host(d_out, r2.out_bytes) == rout
            assert_partial(rerr, args)
        # large: 3 queries x 10^5 alignments + 1.2 M records over 300 k other queries
        rnd = random.Random(3)
        parts = [run_case(100000, rnd, name="contig_%d" % k) for k in range(3)]
        big, _ = H.gen_filter_case(93, n_records=1200000, n_queries=300000)
        text = b"".join(parts) + big
        n_records = text.count(b"\n")
        t0 = time.time()
        rc, out, err = ref_gaffilter(text, ["-r", "2"])
        oracle_s = time.time() - t0
        res_out, res = cv.filter_host(text, g2p.Converter.filter_params(ratio=2))
        assert rc == 0 and g2p.exit_code(res) == 0
        assert res_out == out
        assert "[gaffilter]: filtered %d / %d. total block lengths filtered: %d" % (res.n_filtered, res.n_loaded, res.filtered_len) == last_line(err)
        assert_partial(err, "large")
        print("large gaffilter run: %d records, checker %.1f s" % (n_records, oracle_s))
        assert oracle_s < 120
    finally:
        cv.close()
