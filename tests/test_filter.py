"""gaffilter on the device (SURVEY.md §8f N1; csrc/g2p_filter.cuh) against the reference gaffilter (oracle/_ref/gaffilter,
built unmodified by oracle/build_ref.sh): same kept records, same re-serialisation (tags in name order), same
"[gaffilter]: ..." stderr counts, in GAF and in PAF (-p) mode.  CPU tests run the product kernels under the SIMT
emulator (build/g2p_filter_simt); the GPU tests go through the C-ABI and the drop-in executable, and without the
reference build they compare with its runs stored in tests/golden/reference_runs.json."""
import functools
import hashlib
import json
import os
import subprocess
import tempfile

import pytest

import helpers as H

SIMT = os.path.join(H.BUILD, "g2p_filter_simt")
REF = os.path.join(H.REF_BIN, "gaffilter")
# set by tests/golden/make_reference_runs.py: a file that ref_gaffilter appends its runs to
RECORD = os.environ.get("G2P_RECORD_GAFFILTER")

OPTION_SETS = [
    ["-r", "2"],
    ["-r", "5", "-m", "0.25"],
    ["-o", "100"],
    ["-r", "3", "-q", "5", "-b", "50"],
    ["-r", "2", "-o", "200", "-m", "0.1"],
    ["-r", "1.5", "-i", "1.01"],
]


def simt(text, args):
    p = subprocess.run([SIMT] + args + ["-"], input=text, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return p.returncode, p.stdout, p.stderr.decode("latin-1")


def last_line(err):
    return err.strip().split("\n")[-1]


def md5(data):
    return hashlib.md5(data).hexdigest()


@functools.lru_cache(maxsize=None)
def stored_runs():
    return H.golden("reference_runs.json")["gaffilter_inputs"]


def ref_gaffilter(text, args):
    """(exit code, md5 of stdout, last stderr line) of the reference gaffilter on `text` with `args`: the reference build
    when present, else the run stored in tests/golden/reference_runs.json under the md5 of `text` and `args`."""
    key = "%s %s" % (md5(text), " ".join(args))
    if os.path.exists(REF):
        rc, out, err = H.run_gaffilter_ref(text, args)
    elif RECORD:   # the recording tool was asked to record this project's kernels (see its --source)
        rc, out, err = simt(text, args)
    else:
        if key not in stored_runs():
            raise KeyError("no stored gaffilter run for %s: add it with tests/golden/make_reference_runs.py" % key)
        r = stored_runs()[key]
        return r["rc"], r["md5"], r["err"]
    if RECORD:
        with open(RECORD, "a") as f:
            f.write(json.dumps({"key": key, "rc": rc, "md5": md5(out), "err": last_line(err)}) + "\n")
    return rc, md5(out), last_line(err)


def reference_filter(case, args, text, path=None):
    """(exit code, md5 of stdout, stderr) of the reference gaffilter on `text` = H.gen_filter_case(*case), read from the
    file `path` where `args` says {A}, else from stdin: the reference build when present, else the run stored in
    tests/golden/reference_runs.json (the outputs are megabytes)."""
    if os.path.exists(REF):
        rc, out, err = H.run_tool(REF, [path if a == "{A}" else a for a in args], None if "{A}" in args else text)
        return rc, md5(out), err
    for r in H.golden("reference_runs.json")["gaffilter"]:
        if r["case"] == list(case) and r["args"] == list(args):
            return r["rc"], r["md5"], r["err"]
    raise KeyError("no stored gaffilter run for %r %r: add it to tests/golden/make_reference_runs.py" % (case, args))


@pytest.mark.parametrize("paf", [False, True])
@pytest.mark.parametrize("n_queries", [40, 2500])
def test_emulated_filter_matches_reference(paf, n_queries):
    text, lengths = H.gen_filter_case(11 + n_queries, n_records=2500, n_queries=n_queries, paf=paf)
    for args in OPTION_SETS:
        a = args + (["-p"] if paf else [])
        rc, out, err = ref_gaffilter(text, a)
        src, sout, serr = simt(text, a)
        assert rc == src == 0
        assert md5(sout) == out, a
        assert last_line(serr) == err, a


def test_emulated_filter_edge_cases():
    # empty query intervals, '*' columns, a record alone on its query, duplicate tags in PAF mode, an unterminated last line
    gaf = (b"q1\t100\t10\t10\t+\t>a\t50\t0\t10\t10\t10\t60\ttp:A:P\tcg:Z:10M\n"
           b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60\ttp:A:P\tcg:Z:35M\n"
           b"q1\t100\t9\t11\t-\t>b\t50\t0\t2\t2\t2\t3\ttp:A:S\tcg:Z:2M\n"
           b"q2\t*\t0\t40\t+\t>a\t50\t0\t40\t*\t*\t255\tcg:Z:40M\n"
           b"*\t>s43\t97\t12\t0\t6\t92\n"
           b"q3\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40\t0\tzz:Z:x\taa:i:1\tcg:Z:40M")
    for args in (["-r", "2"], ["-o", "5"], ["-r", "2", "-m", "0.5"]):
        rc, out, err = ref_gaffilter(gaf, args)
        src, sout, serr = simt(gaf, args)
        assert rc == src == 0 and md5(sout) == out and last_line(serr) == err, args
    paf = (b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60\ttp:A:P\tgl:i:35\tgm:i:30\ttp:A:S\tcg:Z:35M\n"
           b"q1\t100\t9\t31\t-\tb\t50\t0\t22\t20\t22\t60\tcg:Z:22M\ttp:A:P\n")
    rc, out, err = ref_gaffilter(paf, ["-p", "-r", "1.2"])
    src, sout, serr = simt(paf, ["-p", "-r", "1.2"])
    assert rc == src == 0 and md5(sout) == out and last_line(serr) == err
    # malformed lines: the reference dies while loading (nothing printed)
    for bad in (gaf.replace(b"q2\t*\t0", b"q2\t\t0"), b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60\n"):
        mode = ["-p"] if bad.startswith(b"q1\t100\t5\t40\t+\ta") else []
        rc, out, err = ref_gaffilter(bad, mode + ["-r", "2"])
        src, sout, serr = simt(bad, mode + ["-r", "2"])
        assert rc == src == 134 and sout == b"" and out == md5(b"")


def test_emulated_filter_large_groups():
    """A few query sequences with thousands of alignments each (assembly contigs): the backward scan is bounded by the
    running maximum of the interval ends."""
    text, lengths = H.gen_filter_case(77, n_records=6000, n_queries=3, paf=False)
    for args in (["-r", "2"], ["-o", "300"]):
        rc, out, err = ref_gaffilter(text, args)
        src, sout, serr = simt(text, args)
        assert rc == src == 0 and md5(sout) == out and last_line(serr) == err


@pytest.mark.gpu
@pytest.mark.parametrize("paf", [False, True])
def test_gpu_filter_matches_reference(g2p, paf):
    import torch
    case = (21, 60000, 4000, paf)
    text, lengths = H.gen_filter_case(*case)
    cv = g2p.Converter(0)
    try:
        for args, kw in ((["-r", "2"], dict(ratio=2)), (["-r", "5", "-m", "0.25", "-q", "5"], dict(ratio=5, min_overlap=0.25, min_mapq=5)),
                         (["-o", "150", "-b", "60"], dict(min_overlap_length=150, min_block_length=60))):
            a = args + (["-p"] if paf else []) + ["-"]
            rc, ref, err = reference_filter(case, a, text)
            out, res = cv.filter_host(text, g2p.Converter.filter_params(paf=paf, **kw))
            assert rc == 0 and res.rec_status == 0
            assert md5(out) == ref, a
            assert "[gaffilter]: filtered %d / %d. total block lengths filtered: %d" % (res.n_filtered, res.n_loaded, res.filtered_len) == last_line(err)
        if paf:
            # gaf2paf -> gaffilter -p with the PAF never leaving the device
            gaf, lengths = H.gen_filter_case(21, n_records=60000, n_queries=4000, paf=False)
            assert cv.load_lengths(lengths)
            t = torch.empty(len(gaf) + 16, dtype=torch.uint8, device="cuda")
            g2p.copy_to_device(t.data_ptr(), gaf)
            torch.cuda.synchronize()
            d_paf, r1 = cv.convert_device(t.data_ptr(), len(gaf), torch.cuda.current_stream().cuda_stream)
            assert g2p.exit_code(r1) == 0
            d_out, r2 = cv.filter_device(d_paf, r1.out_bytes, g2p.Converter.filter_params(paf=True, ratio=2), torch.cuda.current_stream().cuda_stream)
            rc, ref, err = reference_filter(case, ["-r", "2", "-p", "-"], text)
            assert md5(g2p.copy_to_host(d_out, r2.out_bytes)) == ref
    finally:
        cv.close()


@pytest.mark.gpu
def test_gpu_gaffilter_cli(g2p):
    exe = os.path.join(g2p.BIN_DIR, "gaffilter")
    case = (31, 20000, 900, False)
    text, lengths = H.gen_filter_case(*case)
    with tempfile.TemporaryDirectory() as td:
        gp = os.path.join(td, "in.gaf")
        open(gp, "wb").write(text)
        subst = {"{A}": gp}
        for args in (["-r", "2", "{A}"], ["{A}", "-r", "5", "-m", "0.25"], ["-o", "100", "-"]):
            stdin = text if args[-1] == "-" else None
            rc, out, err = H.run_tool(exe, [subst.get(a, a) for a in args], stdin)
            rrc, rout, rerr = reference_filter(case, args, text, gp)
            assert rc == rrc == 0 and md5(out) == rout and err == rerr
        for args in ([], ["{A}"], ["-r", "2"], ["-r", "2", "/nonexistent.gaf"], ["--bogus"]):
            rc, out, err = H.run_tool(exe, [subst.get(a, a) for a in args])
            rrc, rout, rerr = H.reference_cli("gaffilter", args, subst)
            assert rc == rrc and out == rout and err.replace(exe, "X") == rerr


def test_emulated_filter_many_tags():
    """More optional fields than the emit kernels collect (16: the text is rescanned then), repeated names in PAF mode
    (the last one is printed) among and beyond the collected ones, long names."""
    many = [("%c%c:i:%d" % (97 + i // 5, 97 + i % 5, i)).encode() for i in range(22)]
    gaf = b"\n".join([
        b"\t".join([b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60"] + many[:16][::-1] + [b"cg:Z:35M"]),
        b"\t".join([b"q1\t100\t50\t90\t+\t>a\t50\t0\t40\t40\t40\t60"] + many[::-1] + [b"cg:Z:40M", b"longname:Z:v"]),
        b"\t".join([b"q2\t100\t0\t40\t-\t>b\t50\t0\t40\t40\t40\t60", b"tp:A:P", b"cg:Z:40M"]),
    ]) + b"\n"
    rc, out, err = ref_gaffilter(gaf, ["-r", "2"])
    src, sout, serr = simt(gaf, ["-r", "2"])
    assert rc == src == 0 and md5(sout) == out and sout.count(b"\n") == 3 and last_line(serr) == err
    paf = b"\n".join([
        b"\t".join([b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60"] + many[:10] + [b"ac:i:99", b"cg:Z:35M", b"ab:Z:again"]),
        b"\t".join([b"q1\t100\t50\t90\t+\ta\t50\t0\t40\t40\t40\t60"] + many + [b"ab:i:77", b"ea:i:78", b"cg:Z:40M", b"cg:Z:39M1X"]),
        b"\t".join([b"q2\t100\t0\t40\t-\tb\t50\t0\t40\t40\t40\t60", b"cg:Z:40M"]),
    ]) + b"\n"
    rc, out, err = ref_gaffilter(paf, ["-p", "-r", "2"])
    src, sout, serr = simt(paf, ["-p", "-r", "2"])
    assert rc == src == 0 and md5(sout) == out and sout.count(b"\n") == 3 and last_line(serr) == err


def test_emulated_filter_reference_quirks():
    """Found by tests/fuzz_filter_vs_ref.py: the assertions of the reference's filter loop (identity >= 0 on every
    visited interval, oend >= ostart in overlap_size) abort it; path steps are printed from their parsed form; negative
    query starts are accepted; the summed block length is a signed 64-bit number."""
    base = (b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60\ttp:A:P\tcg:Z:35M\n"
            b"q1\t100\t9\t31\t-\t>b\t50\t0\t22\t20\t22\t60\ttp:A:P\tcg:Z:22M\n"
            b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40\t60\tcg:Z:40M\n")
    cases = [
        (base.replace(b"\t20\t22\t60", b"\t-20\t22\t60"), ["-r", "2"]),                     # matches < 0: identity < 0
        (base.replace(b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40", b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t-4\t40"), ["-o", "5"]),   # ... on a record alone on its query
        (base.replace(b"q1\t100\t9\t31", b"q1\t100\t39\t7"), ["-r", "2"]),                  # inverted interval: oend < ostart
        (base.replace(b">b\t", b">b:007-10:9<c: 2-8\t"), ["-r", "2"]),                      # steps re-serialised
        (base.replace(b"q1\t100\t9\t31", b"q1\t100\t-9\t31"), ["-r", "2"]),                 # negative query start
        (base.replace(b"q1\t100\t9\t31", b"q1\t100\t-9\t-3"), ["-o", "3"]),
        (base.replace(b"\t20\t22\t60", b"\t20\t9223372036854775807\t60").replace(b"35\t35\t35\t60", b"35\t35\t9223372036854775800\t60"), ["-r", "1.0001"]),
    ]
    for data, args in cases:
        rc, out, err = ref_gaffilter(data, args)
        src, sout, serr = simt(data, args)
        assert src == rc, (data, args)
        if rc == 0:
            assert md5(sout) == out and last_line(serr) == err, (data, args)
        else:
            assert sout == b""
