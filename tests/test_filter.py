"""gaffilter on the device (SURVEY.md §8f N1; csrc/g2p_filter.cuh) against the reference gaffilter: same kept records,
same re-serialisation (tags in name order), same "[gaffilter]: ..." stderr counts, in GAF and in PAF (-p) mode.  The
checker is the reference build (oracle/_ref/gaffilter, built unmodified by oracle/build_ref.sh) when present, else the
independent restatement oracle/bin/gaffilter_oracle, which tests/golden/reference_runs.json pins
(test_gaffilter_oracle_reproduces_stored_runs).  CPU tests run the product kernels under the SIMT emulator
(build/g2p_filter_simt); the GPU tests go through the C-ABI and the drop-in executable.  Every differential case filters
some records and keeps others."""
import hashlib
import os
import re
import subprocess
import tempfile

import pytest

import helpers as H

SIMT = os.path.join(H.BUILD, "g2p_filter_simt")
REF = os.path.join(H.REF_BIN, "gaffilter")

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


def checker():
    """The gaffilter the kernels are compared with: the reference build when present, else the restatement."""
    return H.oracle_path("auto", "gaffilter")[0]


def ref_gaffilter(text, args):
    """(exit code, stdout, stderr) of the reference gaffilter (or its restatement) on `text` with `args`."""
    return H.run_tool(checker(), list(args) + ["-"], text)


def reference_filter(case, args, text, path=None):
    """(exit code, md5 of stdout, stderr) of the reference gaffilter (or its restatement) on `text` =
    H.gen_filter_case(*case), read from the file `path` where `args` says {A}, else from stdin."""
    rc, out, err = H.run_tool(checker(), [path if a == "{A}" else a for a in args], None if "{A}" in args else text)
    return rc, md5(out), err


def counts(err):
    """(filtered, loaded) of the summary line."""
    m = re.search(r"\[gaffilter\]: filtered (\d+) / (\d+)\.", last_line(err))
    assert m, err
    return int(m.group(1)), int(m.group(2))


def assert_partial(err, what=""):
    """The run filtered some records and kept others: a kernel that kept or dropped everything would not pass."""
    filtered, loaded = counts(err)
    assert 0 < filtered < loaded, (what, filtered, loaded)


def same_as_reference(text, args, partial=True):
    """The emulated kernels and the checker agree on `text`: exit code, stdout bytes, summary line."""
    rc, out, err = ref_gaffilter(text, args)
    src, sout, serr = simt(text, args)
    assert src == rc, (args, rc, src, serr[-300:])
    if rc == 0:
        assert sout == out, args
        assert last_line(serr) == last_line(err), args
        if partial:
            assert_partial(err, args)
    else:
        assert sout == b"" and out == b"", args
    return rc, out, err


# ---- inputs of the emulator tests ---------------------------------------------------------------------------------
# empty query intervals, '*' columns, a record alone on its query, duplicate tags in PAF mode, an unterminated last line
EDGE_GAF = (b"q1\t100\t10\t10\t+\t>a\t50\t0\t10\t10\t10\t60\ttp:A:P\tcg:Z:10M\n"
            b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60\ttp:A:P\tcg:Z:35M\n"
            b"q1\t100\t9\t11\t-\t>b\t50\t0\t2\t2\t2\t3\ttp:A:S\tcg:Z:2M\n"
            b"q2\t*\t0\t40\t+\t>a\t50\t0\t40\t*\t*\t255\tcg:Z:40M\n"
            b"*\t>s43\t97\t12\t0\t6\t92\n"
            b"q3\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40\t0\tzz:Z:x\taa:i:1\tcg:Z:40M")
EDGE_GAF_ARGS = (["-r", "2"], ["-o", "5"], ["-r", "2", "-m", "0.5"])
EDGE_PAF = (b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60\ttp:A:P\tgl:i:35\tgm:i:30\ttp:A:S\tcg:Z:35M\n"
            b"q1\t100\t9\t31\t-\tb\t50\t0\t22\t20\t22\t60\tcg:Z:22M\ttp:A:P\n")
# malformed lines: the reference dies while loading (nothing printed)
EDGE_BAD = ((EDGE_GAF.replace(b"q2\t*\t0", b"q2\t\t0"), ["-r", "2"]), (b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60\n", ["-p", "-r", "2"]))
MANY = [("%c%c:i:%d" % (97 + i // 5, 97 + i % 5, i)).encode() for i in range(22)]
MANY_TAGS_GAF = b"\n".join([
    b"\t".join([b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60"] + MANY[:16][::-1] + [b"cg:Z:35M"]),
    b"\t".join([b"q1\t100\t50\t90\t+\t>a\t50\t0\t40\t40\t40\t60"] + MANY[::-1] + [b"cg:Z:40M", b"longname:Z:v"]),
    b"\t".join([b"q2\t100\t0\t40\t-\t>b\t50\t0\t40\t40\t40\t60", b"tp:A:P", b"cg:Z:40M"]),
]) + b"\n"
MANY_TAGS_PAF = b"\n".join([
    b"\t".join([b"q1\t100\t5\t40\t+\ta\t50\t0\t35\t35\t35\t60"] + MANY[:10] + [b"ac:i:99", b"cg:Z:35M", b"ab:Z:again"]),
    b"\t".join([b"q1\t100\t50\t90\t+\ta\t50\t0\t40\t40\t40\t60"] + MANY + [b"ab:i:77", b"ea:i:78", b"cg:Z:40M", b"cg:Z:39M1X"]),
    b"\t".join([b"q2\t100\t0\t40\t-\tb\t50\t0\t40\t40\t40\t60", b"cg:Z:40M"]),
]) + b"\n"
# a secondary record under the primary one of q2: filtered with -r 2, so that the tag tests also see a record dropped
MANY_TAGS_EXTRA_GAF = b"q2\t100\t2\t30\t+\t>c\t50\t0\t28\t28\t28\t60\ttp:A:S\t" + b"\t".join(MANY[3:19]) + b"\tcg:Z:28M\n"
MANY_TAGS_EXTRA_PAF = b"q2\t100\t2\t30\t+\tc\t50\t0\t28\t28\t28\t60\ttp:A:S\t" + b"\t".join(MANY[3:19]) + b"\tcg:Z:28M\ttp:A:P\ttp:A:S\n"
QUIRK_BASE = (b"q1\t100\t5\t40\t+\t>a\t50\t0\t35\t35\t35\t60\ttp:A:P\tcg:Z:35M\n"
              b"q1\t100\t9\t31\t-\t>b\t50\t0\t22\t20\t22\t60\ttp:A:P\tcg:Z:22M\n"
              b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40\t60\tcg:Z:40M\n")
QUIRKS = [
    (QUIRK_BASE.replace(b"\t20\t22\t60", b"\t-20\t22\t60"), ["-r", "2"]),                     # matches < 0: identity < 0
    (QUIRK_BASE.replace(b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t40\t40", b"q2\t100\t0\t40\t+\t>a\t50\t0\t40\t-4\t40"), ["-o", "5"]),   # ... alone on its query
    (QUIRK_BASE.replace(b"q1\t100\t9\t31", b"q1\t100\t39\t7"), ["-r", "2"]),                  # inverted interval: oend < ostart
    (QUIRK_BASE.replace(b">b\t", b">b:007-10:9<c: 2-8\t"), ["-r", "2"]),                      # steps re-serialised
    (QUIRK_BASE.replace(b"q1\t100\t9\t31", b"q1\t100\t-9\t31"), ["-r", "2"]),                 # negative query start
    (QUIRK_BASE.replace(b"q1\t100\t9\t31", b"q1\t100\t-9\t-3"), ["-o", "3"]),
    (QUIRK_BASE.replace(b"\t20\t22\t60", b"\t20\t9223372036854775807\t60").replace(b"35\t35\t35\t60", b"35\t35\t9223372036854775800\t60"), ["-r", "1.0001"]),
]


def stored_inputs():
    """(text, args) of every gaffilter run in tests/golden/reference_runs.json "gaffilter_inputs" (keyed by the md5 of
    the text and the arguments): the inputs the emulator tests used when the file was recorded."""
    for paf in (False, True):
        for n_queries in (40, 2500):
            text, _ = H.gen_filter_case(11 + n_queries, n_records=2500, n_queries=n_queries, paf=paf)
            for args in OPTION_SETS:
                yield text, args + (["-p"] if paf else [])
    for args in EDGE_GAF_ARGS:
        yield EDGE_GAF, args
    yield EDGE_PAF, ["-p", "-r", "1.2"]
    for text, args in EDGE_BAD:
        yield text, args
    text, _ = H.gen_filter_case(77, n_records=6000, n_queries=3, paf=False)
    for args in (["-r", "2"], ["-o", "300"]):
        yield text, args
    yield MANY_TAGS_GAF, ["-r", "2"]
    yield MANY_TAGS_PAF, ["-p", "-r", "2"]
    for text, args in QUIRKS:
        yield text, args


def test_gaffilter_oracle_reproduces_stored_runs():
    """The restatement oracle/bin/gaffilter_oracle reproduces every stored gaffilter run: exit code, stdout md5, summary
    line (41 emulator-test inputs) or whole stderr (9 generator cases of the GPU tests)."""
    port, kind = H.oracle_path("port", "gaffilter")
    stored = H.golden("reference_runs.json")
    seen = set()
    for text, args in stored_inputs():
        key = "%s %s" % (md5(text), " ".join(args))
        r = stored["gaffilter_inputs"][key]
        rc, out, err = H.run_tool(port, args + ["-"], text)
        assert (rc, md5(out)) == (r["rc"], r["md5"]), key
        if rc == 0:
            assert last_line(err) == r["err"], key
        seen.add(key)
    assert seen == set(stored["gaffilter_inputs"]) and len(seen) == 41
    assert len(stored["gaffilter"]) == 9
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "in.gaf")
        for r in stored["gaffilter"]:
            text, _ = H.gen_filter_case(*r["case"])
            open(path, "wb").write(text)
            args = [path if a == "{A}" else a for a in r["args"]]
            rc, out, err = H.run_tool(port, args, None if "{A}" in r["args"] else text)
            assert (rc, md5(out), len(out), err) == (r["rc"], r["md5"], r["bytes"], r["err"]), r["args"]


def test_gaffilter_oracle_reproduces_quirks():
    """The quirks the reference fuzzing found, restated: its filter-loop assertions abort (identity < 0 on any visited
    interval, the record's own included; oend < ostart), path steps print from their parsed form, negative starts load."""
    port, kind = H.oracle_path("port", "gaffilter")
    expect = [134, 134, 134, 0, 0, 0, 0]
    for (text, args), want in zip(QUIRKS, expect):
        rc, out, err = H.run_tool(port, args + ["-"], text)
        assert rc == want, (text, args, err)
        if rc:
            assert out == b""
    rc, out, err = H.run_tool(port, ["-o", "100", "-"], QUIRKS[3][0])
    assert b">b:7-10<c:2-8\t" in out


@pytest.mark.skipif(not os.path.exists(REF), reason="needs the reference build oracle/_ref/gaffilter")
@pytest.mark.parametrize("seed", [1, 2])
def test_gaffilter_oracle_differential(seed):
    """Seeded differential runs of the restatement against the reference build (the pin of the port)."""
    import random
    rnd = random.Random(seed)
    port, kind = H.oracle_path("port", "gaffilter")
    for it in range(12):
        paf = it % 2 == 1
        text, _ = H.gen_filter_case(seed * 1000 + it, n_records=rnd.choice([300, 2000]), n_queries=rnd.choice([20, 200, 1000]), paf=paf)
        args = rnd.choice(OPTION_SETS) + (["-p"] if paf else [])
        got = H.run_tool(port, args + ["-"], text)
        ref = H.run_tool(REF, args + ["-"], text)
        assert got[0] == ref[0] and got[1] == ref[1], args
        if ref[0] == 0:
            assert last_line(got[2]) == last_line(ref[2])


@pytest.mark.parametrize("paf", [False, True])
@pytest.mark.parametrize("n_queries", [40, 2500])
def test_emulated_filter_matches_reference(paf, n_queries):
    # about six records per query sequence: every option set filters some records and keeps others
    text, lengths = H.gen_filter_case(11 + n_queries, n_records=min(2500, 6 * n_queries), n_queries=n_queries, paf=paf)
    for args in OPTION_SETS:
        same_as_reference(text, args + (["-p"] if paf else []))


def test_emulated_filter_edge_cases():
    for args in EDGE_GAF_ARGS:
        same_as_reference(EDGE_GAF, args)
    same_as_reference(EDGE_PAF, ["-p", "-r", "1.2"], partial=False)   # (two records: -r 1.2 filters one of them)
    for bad, args in EDGE_BAD:
        rc, out, err = same_as_reference(bad, args)
        assert rc == 134


def test_emulated_filter_large_groups():
    """A few query sequences with thousands of alignments each, spread along them (assembly contigs): the backward scan
    is bounded by the running maximum of the interval ends, runs cross the 2048-entry tiles of the sort and the scan."""
    text = H.gen_spread_filter_case(77, n_records=6000, n_queries=3)
    for args in (["-r", "2"], ["-o", "300"], ["-r", "3", "-m", "0.5", "-q", "5"]):
        same_as_reference(text, args)


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
            assert_partial(err, a)
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
            assert_partial(err, args)
        for args in ([], ["{A}"], ["-r", "2"], ["-r", "2", "/nonexistent.gaf"], ["--bogus"]):
            rc, out, err = H.run_tool(exe, [subst.get(a, a) for a in args])
            rrc, rout, rerr = H.reference_cli("gaffilter", args, subst)
            assert rc == rrc and out == rout and err.replace(exe, "X") == rerr


def test_emulated_filter_many_tags():
    """More optional fields than the emit kernels collect (16: the text is rescanned then), repeated names in PAF mode
    (the last one is printed) among and beyond the collected ones, long names."""
    rc, out, err = same_as_reference(MANY_TAGS_GAF + MANY_TAGS_EXTRA_GAF, ["-r", "2"])
    assert out.count(b"\n") == 3
    rc, out, err = same_as_reference(MANY_TAGS_PAF + MANY_TAGS_EXTRA_PAF, ["-p", "-r", "2"])
    assert out.count(b"\n") == 3


def test_emulated_filter_reference_quirks():
    """Found by tests/fuzz_filter_vs_ref.py: the assertions of the reference's filter loop (identity >= 0 on every
    visited interval, oend >= ostart in overlap_size) abort it; path steps are printed from their parsed form; negative
    query starts are accepted; the summed block length is a signed 64-bit number."""
    for i, (data, args) in enumerate(QUIRKS):
        if i == 5:   # (records below 0 only: one more, inside the negative one, so that -o 3 filters something)
            data += b"q1\t100\t-6\t-4\t+\t>a\t50\t0\t2\t2\t2\t60\tcg:Z:2M\n"
        same_as_reference(data, args)
