"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the
C-ABI of libg2p.so; the CPU oracle (oracle/_ref reference build when present, else the
restatement) is only the checker.  Bar: byte-identical PAF, same exit code, same stderr
line for the reference's exit(1) errors."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import pytest

import helpers as H

pytestmark = pytest.mark.gpu


def test_native_library_is_what_runs(g2p, converter):
    """The extension in-tree is loaded and a conversion launches kernels."""
    maps = open("/proc/self/maps").read()
    assert "libg2p.so" in maps
    d = H.golden("gaf2paf_kat.json")
    assert converter.load_lengths(d["lengths"].encode())
    out, res = converter.convert_host((d["vectors"][0]["in"] + "\n").encode("latin-1"))
    assert res.gpu_launches >= 2
    assert out.decode("latin-1") == d["vectors"][0]["out"]


def test_golden_vectors(g2p, converter):
    d = H.golden("gaf2paf_kat.json")
    assert converter.load_lengths(d["lengths"].encode())
    for v in d["vectors"]:
        gaf = (v["in"] + "\n").encode("latin-1")
        out, res = converter.convert_host(gaf)
        rc = g2p.exit_code(res)
        assert rc == v["rc"], v["name"]
        if rc != 134:
            assert out.decode("latin-1") == v["out"], v["name"]
        if rc == 1:
            assert g2p.Converter.format_error(res, gaf) == v["err"], v["name"]
    out, res = converter.convert_host(("\n".join(d["stream"]["in"]) + "\n").encode("latin-1"))
    assert g2p.exit_code(res) == 0 and out.decode("latin-1") == d["stream"]["out"]
    # unterminated last line
    out, res = converter.convert_host("\n".join(d["stream"]["in"]).encode("latin-1"))
    assert g2p.exit_code(res) == 0 and out.decode("latin-1") == d["stream"]["out"]


def test_error_in_the_middle_keeps_earlier_output(g2p, converter):
    d = H.golden("gaf2paf_kat.json")
    assert converter.load_lengths(d["lengths"].encode())
    vec = {v["name"]: v for v in d["vectors"]}
    good = [v for v in d["vectors"] if v["rc"] == 0 and v["out"]]
    for bad_name in ("X7-unknown-name-second-step-partial-output", "K21-no-cg-exit1", "K19-cigar-too-short-abort"):
        bad = vec[bad_name]
        head = good[:40]
        lines = [g["in"] for g in head] + [bad["in"]] + [g["in"] for g in good[:5]]
        gaf = ("\n".join(lines) + "\n").encode("latin-1")
        out, res = converter.convert_host(gaf)
        rc, ref_out, ref_err, kind = H.run_gaf2paf_cpu(gaf, d["lengths"].encode())
        assert g2p.exit_code(res) == rc == bad["rc"]
        assert res.err_record == len(head)
        if rc == 1:
            assert out == ref_out
            assert g2p.Converter.format_error(res, gaf) == ref_err
        else:
            assert out.decode("latin-1") == "".join(g["out"] for g in head)


def test_empty_and_degenerate_inputs(g2p, converter):
    d = H.golden("gaf2paf_kat.json")
    assert converter.load_lengths(d["lengths"].encode())
    out, res = converter.convert_host(b"")
    assert out == b"" and res.n_records == 0 and g2p.exit_code(res) == 0
    out, res = converter.convert_host(b"*\t>s43\t97\t12\t0\t6\t92\n" * 3)
    assert out == b"" and res.n_records == 3 and g2p.exit_code(res) == 0
    out, res = converter.convert_host(b"\n")           # blank line: the reference aborts in parse_gaf_record
    assert g2p.exit_code(res) == 134


@pytest.mark.parametrize("name,count,over", [
    ("short", 200000, {"pct_star": 2}),
    ("short_eqx", 50000, {}),
    ("stable", 3000, {}),
    ("medium", 3000, {}),
    ("asm", 24, {}),
    ("asm", 3, {"steps_lo": 30000, "steps_hi": 40000}),
])
def test_synthetic_parity(g2p, name, count, over):
    p = H.preset(name, seed=21, **over)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, count)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out, res = cv.convert_host(gaf)
    finally:
        cv.close()
    rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0 and g2p.exit_code(res) == 0
    assert res.n_records == gaf.count(b"\n")
    assert len(out) == len(ref)
    assert out == ref, "PAF differs from the %s oracle" % kind


def test_mixed_skew_parity(g2p):
    """Short and assembly-scale records interleaved in one buffer (config 5 shape)."""
    ps, pa = H.preset("short", seed=31), H.preset("asm", seed=31, n_nodes=200000, node_len_lo=20, node_len_hi=400)
    lengths = H.gen_lengths(ps)    # same node-length function and seed -> one table serves both
    parts = []
    for i in range(6):
        parts.append(H.gen_records(ps, i * 5000, 5000))
        parts.append(H.gen_records(pa, i, 1))
    gaf = b"".join(parts)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out, res = cv.convert_host(gaf)
    finally:
        cv.close()
    rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0 and g2p.exit_code(res) == 0 and out == ref


def test_sharded_equals_whole(g2p):
    """Newline-aligned byte-range shards converted independently and concatenated in
    order reproduce the unsharded output (the multi-GPU scheme, on one device)."""
    p = H.preset("short", seed=41)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, 60000)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        whole, res = cv.convert_host(gaf)
        for n in (2, 3, 8):
            parts = [cv.convert_host(gaf[a:b])[0] for a, b in g2p.shard_ranges(gaf, n)]
            assert b"".join(parts) == whole
    finally:
        cv.close()


def test_full_size_properties(g2p):
    """BASELINE config 3 scale (reduced to what one test may take): properties that do not
    need the oracle — determinism, line accounting, and a sampled slice checked exactly."""
    import torch
    p = H.preset("short", seed=51)
    lengths = H.gen_lengths(p)
    count = 2_000_000
    gaf = H.gen_records(p, 0, count)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out1, res1 = cv.convert_host(gaf)
        out2, res2 = cv.convert_host(gaf)
        assert res1.n_records == count and g2p.exit_code(res1) == 0
        assert hashlib.md5(out1).digest() == hashlib.md5(out2).digest()
        assert out1.endswith(b"\n")
        # every PAF line carries the 12 columns + gm/gl/gi/cg tags
        sample = out1[:2_000_000]
        for line in sample.split(b"\n")[:-1][:2000]:
            f = line.split(b"\t")
            assert len(f) >= 16 and f[-1].startswith(b"cg:Z:") and f[4] in (b"+", b"-")
        # sampled newline-aligned slice against the oracle
        a, b = g2p.shard_ranges(gaf, 200)[77]
        rc, ref, err, kind = H.run_gaf2paf_cpu(gaf[a:b], lengths)
        got, r = cv.convert_host(gaf[a:b])
        assert rc == 0 and got == ref
    finally:
        cv.close()


def test_device_resident_entry_point(g2p):
    import torch
    p = H.preset("short", seed=61)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, 30000)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        t = torch.empty(len(gaf) + 16, dtype=torch.uint8, device="cuda")
        g2p.copy_to_device(t.data_ptr(), gaf)
        torch.cuda.synchronize()
        d_out, res = cv.convert_device(t.data_ptr(), len(gaf), torch.cuda.current_stream().cuda_stream)
        ref_out, _ = cv.convert_host(gaf)
        assert g2p.copy_to_host(d_out, res.out_bytes) == ref_out
        # line index on its own
        starts, nl = cv.index_lines(t.data_ptr(), len(gaf), torch.cuda.current_stream().cuda_stream)
        assert nl == 30000
        import numpy as np
        got = np.frombuffer(g2p.copy_to_host(starts, 4 * (nl + 1)), dtype=np.uint32)
        exp = np.flatnonzero(np.frombuffer(gaf, dtype=np.uint8) == 10) + 1
        assert got[0] == 0 and (got[1:] == exp).all()
    finally:
        cv.close()


def test_cli_end_to_end(g2p):
    """The drop-in executable: same stdout / exit code as the CPU oracle, incl. stdin and two files."""
    exe = os.path.join(g2p.BIN_DIR, "gaf2paf")
    p = H.preset("short", seed=71)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, 20000)
    binary, kind = H.oracle_path()
    with tempfile.TemporaryDirectory() as td:
        lp, a, b = os.path.join(td, "l.tsv"), os.path.join(td, "a.gaf"), os.path.join(td, "b.gaf")
        open(lp, "wb").write(lengths)
        half = gaf.rfind(b"\n", 0, len(gaf) // 2) + 1
        open(a, "wb").write(gaf[:half - 1])     # first file without trailing newline
        open(b, "wb").write(gaf[half:])
        rc, out, err = H.run_tool(exe, [a, b, "-l", lp])
        rrc, rout, rerr = H.run_tool(binary, [a, b, "-l", lp])
        assert rc == rrc == 0 and out == rout
        rc, out, err = H.run_tool(exe, ["-l", lp, "-"], gaf)
        assert rc == 0 and out == rout
        # small chunks force the newline-aligned carry logic
        env = dict(os.environ, G2P_CHUNK_MB="1")
        pr = subprocess.run([exe, "-l", lp, a, b], stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
        assert pr.returncode == 0 and pr.stdout == rout
        # error path: unknown name -> message + exit 1, earlier output kept
        bad = gaf[:half] + b"q\t100\t0\t15\t+\t>zzz:0-15\t15\t0\t15\t15\t15\t60\tcg:Z:15M\n" + gaf[half:]
        rc, out, err = H.run_tool(exe, ["-", "-l", lp], bad)
        rrc, rout2, rerr = H.run_tool(binary, ["-", "-l", lp], bad)
        assert rc == rrc == 1 and out == rout2 and err == rerr


def test_host_call_pipelines_chunks(g2p, monkeypatch):
    """g2p_convert_host cuts large inputs into newline-aligned chunks driven by several host threads
    (copy/compute overlap).  Force many small chunks and compare with the oracle, with and without
    a failing record in a middle chunk."""
    monkeypatch.setenv("G2P_HOST_CHUNK_MB", "1")
    p = H.preset("short", seed=81, pct_star=1)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, 70000)
    pa = H.preset("asm", seed=81, n_nodes=200000, node_len_lo=20, node_len_hi=400, steps_lo=300, steps_hi=3000)
    mid = gaf.rfind(b"\n", 0, len(gaf) // 2) + 1
    gaf = gaf[:mid] + H.gen_records(pa, 0, 20) + gaf[mid:]
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out, res = cv.convert_host(gaf)
        rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
        assert rc == 0 and g2p.exit_code(res) == 0
        assert res.n_records == gaf.count(b"\n") and out == ref
        # second call reuses the grown buffers
        out2, _ = cv.convert_host(gaf)
        assert out2 == ref
        # failing record in a middle chunk: output up to it, same message, later chunks ignored
        cutp = gaf.rfind(b"\n", 0, len(gaf) * 2 // 3) + 1
        bad = gaf[:cutp] + b"q\t100\t0\t15\t+\t>zzz:0-15\t15\t0\t15\t15\t15\t60\tcg:Z:15M\n" + gaf[cutp:]
        out, res = cv.convert_host(bad)
        rc, ref, err, kind = H.run_gaf2paf_cpu(bad, lengths)
        assert rc == 1 and g2p.exit_code(res) == 1
        assert out == ref and g2p.Converter.format_error(res, bad) == err
        assert res.err_record == gaf[:cutp].count(b"\n")
    finally:
        cv.close()


# ---- gaf2unstable (BASELINE config 2) ------------------------------------------------------
def test_gaf2unstable_golden(g2p):
    d = H.golden("gaf2unstable_kat.json")
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(d["rgfa"].encode())
        assert ok
        assert cv.node_lengths().decode() == d["node_lengths"]
        for v in d["vectors"]:
            out, res, warns = cv.unstable_host((v["in"] + "\n").encode())
            assert g2p.exit_code(res) == v["rc"] and out.decode() == v["out"], v["in"]
        out, res, warns = cv.unstable_host(("\n".join(d["stream"]["in"]) + "\n").encode())
        assert out.decode() == d["stream"]["out"] and res.gpu_launches >= 5
        # second stage on the same context: gaf2paf -l node-lengths
        assert cv.load_lengths(cv.node_lengths())
        paf, res2 = cv.convert_host(out)
        assert paf.decode() == d["paf"]["out"] and g2p.exit_code(res2) == d["paf"]["rc"]
    finally:
        cv.close()


@pytest.mark.parametrize("seed,aligned", [(11, False), (12, True)])
def test_gaf2unstable_synthetic_and_two_stage(g2p, seed, aligned):
    """gaf2unstable on a synthetic rGFA == reference (stdout, -o file, warnings); for node-aligned
    input the two-stage pipeline gaf2unstable | gaf2paf == the reference's (README.md:55-58)."""
    rgfa, gaf = H.gen_rgfa_case(seed, n_records=4000, aligned=aligned)
    rc, ref, err, nl = H.run_gaf2unstable_ref(gaf, rgfa, True)
    assert rc == 0
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(rgfa)
        assert ok and cv.node_lengths() == nl
        out, res, warns = cv.unstable_host(gaf)
        assert g2p.exit_code(res) == 0 and out == ref
        assert "".join(warns) == err
        if aligned:
            rc2, paf_ref, err2, kind = H.run_gaf2paf_cpu(ref, nl)
            assert cv.load_lengths(nl)
            paf, res2 = cv.convert_host(out)
            assert rc2 == 0 and g2p.exit_code(res2) == 0 and paf == paf_ref
    finally:
        cv.close()


@pytest.mark.parametrize("seed", [31, 32])
def test_fused_unstable_convert_equals_the_two_stage_pipeline(g2p, seed):
    """N2 (SURVEY.md §8f): `gaf2unstable in.gaf -g g.gfa -o L | gaf2paf - -l L` as one call whose intermediate GAF stays in
    device memory == the reference's two processes (README.md:55-58), including the stage-1 warnings and a record on
    which the reference's gaf2unstable aborts."""
    import torch
    rgfa, gaf = H.gen_rgfa_case(seed, n_records=6000, aligned=True, multi_ref_pct=4)
    rc, ugaf, err, nl = H.run_gaf2unstable_ref(gaf, rgfa, want_lengths=True)
    rc2, paf_ref, err2, kind = H.run_gaf2paf_cpu(ugaf, nl)
    assert rc == 0 and rc2 == 0
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(rgfa)
        assert ok
        paf, res, warn_text = cv.unstable_convert_host(gaf)
        assert g2p.exit_code(res) == 0 and res.stage == 0
        assert paf == paf_ref
        assert warn_text == err
        assert res.mid_bytes == len(ugaf) and res.unstable_ms > 0
        # device-resident entry point
        t = torch.empty(len(gaf) + 16, dtype=torch.uint8, device="cuda")
        g2p.copy_to_device(t.data_ptr(), gaf)
        torch.cuda.synchronize()
        d_out, res2 = cv.unstable_convert_device(t.data_ptr(), len(gaf), torch.cuda.current_stream().cuda_stream)
        assert g2p.copy_to_host(d_out, res2.out_bytes) == paf_ref
        # the -l table of the context is not touched by the fused call
        p = H.preset("short", seed=3)
        lengths = H.gen_lengths(p)
        g = H.gen_records(p, 0, 2000)
        assert cv.load_lengths(lengths)
        cv.unstable_convert_host(gaf)
        out, r3 = cv.convert_host(g)
        assert out == H.run_gaf2paf_cpu(g, lengths)[1]
        # stage 1 stops at a record (unknown contig: the reference's gaf2unstable aborts): what came before is converted
        lines = gaf.split(b"\n")
        k = len(lines) // 2
        bad = b"\n".join(lines[:k] + [b"q\t100\t0\t15\t+\t>nosuchcontig:0-15\t15\t0\t15\t15\t15\t60\tcg:Z:15M"] + lines[k:])
        paf_b, res_b, _ = cv.unstable_convert_host(bad)
        head = b"\n".join(lines[:k]) + b"\n"
        rc, ugaf_h, err_h, nl_h = H.run_gaf2unstable_ref(head, rgfa, want_lengths=True)
        assert g2p.exit_code(res_b) == 134 and res_b.stage == 1
        assert paf_b == H.run_gaf2paf_cpu(ugaf_h, nl_h)[1]
    finally:
        cv.close()


def test_gaf2unstable_abort_and_cli(g2p):
    rgfa, gaf = H.gen_rgfa_case(21, n_records=1500, aligned=True)
    bad = gaf + b"q\t100\t0\t15\t+\t>nosuchcontig:0-15\t15\t0\t15\t15\t15\t60\tcg:Z:15M\n" + gaf[:2000]
    exe = os.path.join(g2p.BIN_DIR, "gaf2unstable")
    ref_exe, _kind = H.oracle_path("auto", "gaf2unstable")   # the reference build when present, else the restatement
    with tempfile.TemporaryDirectory() as td:
        gp, a = os.path.join(td, "g.gfa"), os.path.join(td, "a.gaf")
        open(gp, "wb").write(rgfa)
        open(a, "wb").write(gaf)
        l1, l2 = os.path.join(td, "l1.tsv"), os.path.join(td, "l2.tsv")
        rc, out, err = H.run_tool(exe, [a, "-g", gp, "-o", l1])
        rrc, rout, rerr = H.run_tool(ref_exe, [a, "-g", gp, "-o", l2])
        assert rc == rrc == 0 and out == rout and err == rerr
        assert open(l1, "rb").read() == open(l2, "rb").read()
        rc, out, err = H.run_tool(exe, ["-", "--rgfa", gp], bad)
        rrc, rout, rerr = H.run_tool(ref_exe, ["-", "--rgfa", gp], bad)
        assert rc == rrc == 134
        assert out == rout[:len(out)]
        assert out.count(b"\n") == sum(1 for ln in gaf.split(b"\n")[:-1] if not ln.startswith(b"*"))   # records before the failing one
        # usage errors
        subst = {"{A}": a, "{G}": gp}
        for args in ([], ["{A}"], ["{A}", "b", "c", "-g", "{G}"]):
            rc, out, err = H.run_tool(exe, [subst.get(x, x) for x in args])
            rrc, rout, rerr = H.reference_cli("gaf2unstable", args, subst)
            assert rc == rrc and err.replace(exe, "X") == rerr


def test_descriptor_overflow_falls_back_to_reparsing_emit(g2p, monkeypatch):
    """A descriptor array that is too small must only cost speed: the records whose lines do not fit
    are emitted by the re-parsing kernels (k_short<true>, k_long<true>)."""
    monkeypatch.setenv("G2P_DESC_CAP", "4096")
    ps = H.preset("short", seed=91)
    pm = H.preset("medium", seed=91)
    lengths = H.gen_lengths(ps)
    gaf = H.gen_records(ps, 0, 20000) + H.gen_records(pm, 0, 300) + H.gen_records(ps, 20000, 5000)
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out, res = cv.convert_host(gaf)
    finally:
        cv.close()
    rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0 and g2p.exit_code(res) == 0 and out == ref


def test_one_pass_index_variant(g2p, monkeypatch):
    """The optional single-pass index (k_index1: TMA tiles + decoupled look-back) gives the same
    result as the default counting kernels; a blank-line flood exercises its capacity fallback."""
    p = H.preset("short", seed=111, pct_star=1)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, 30000)
    monkeypatch.setenv("G2P_ONE_PASS_INDEX", "0")
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out, res = cv.convert_host(gaf)
        out_nonl, _ = cv.convert_host(gaf[:-1])          # unterminated last line
    finally:
        cv.close()
    monkeypatch.setenv("G2P_ONE_PASS_INDEX", "1")
    rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0 and out == ref and out_nonl == ref
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        out1, _ = cv.convert_host(gaf[:-1])
        assert out1 == ref
        flood = gaf[:5000].rsplit(b"\n", 1)[0] + b"\n" * 200000   # far more lines than bytes / 32: reference aborts on the first blank line
        o2, r2 = cv.convert_host(flood)
        rc2, ref2, err2, _ = H.run_gaf2paf_cpu(flood, lengths)
        assert rc2 == 134 and g2p.exit_code(r2) == 134 and r2.n_records == flood.count(b"\n")
        assert o2 == ref2[:len(o2)]
    finally:
        cv.close()


def test_late_delegation(g2p):
    """Long records that k_long delegates after having described some of their lines (non-canonical
    or invalid last CIGAR op), in the middle and at the very end of the buffer."""
    import test_oracle
    lengths, cases = test_oracle._late_cases()
    cv = g2p.Converter(0)
    try:
        assert cv.load_lengths(lengths)
        for name, lines in cases.items():
            data = b"\n".join(lines) + b"\n"
            out, res = cv.convert_host(data)
            rc, ref, err, kind = H.run_gaf2paf_cpu(data, lengths)
            assert g2p.exit_code(res) == rc, name
            assert (out == ref) if rc != 134 else ref.startswith(out), name
    finally:
        cv.close()


@pytest.mark.parametrize("env", [
    {},                                            # default dispatch (k_fuse when it pays, else the two-pass pipeline)
    {"G2P_FUSE": "2"},                             # the one-pass kernel k_fuse first, default configuration (24 KiB tiles, direct stores)
    {"G2P_FUSE": "2", "G2P_FUSE_CFG": "0"},        # 32 KiB tiles, staged lines + TMA bulk store
    {"G2P_FUSE": "2", "G2P_FUSE_CFG": "2"},        # 16 KiB tiles, three CTAs per SM
    {"G2P_FUSE": "2", "G2P_FUSE_CFG": "4", "G2P_FUSE_OUT_CAP": "65536"},   # 8 KiB tiles; the output buffer starts too small: grow and run again
    {"G2P_FUSE": "0"},                             # the general two-pass pipeline alone (k_rec + scans + k_emit_lines)
    {"G2P_FUSE": "0", "G2P_SIZE_KERNEL": "short"},                  # the 8-lanes-per-record size pass
    {"G2P_FUSE": "0", "G2P_LEN_SORT": "1"},                         # k_rec on records ordered by length class
    {"G2P_FUSE": "0", "G2P_REC_CHUNKS": "9"},                       # small k_rec slots: the longer half of the records goes to k_long
    {"G2P_FUSE": "0", "G2P_REC_CHUNKS": "16", "G2P_LEN_SORT": "1"},
])
def test_size_pass_variants(g2p, monkeypatch, env):
    """Every selectable form of the short-record size pass (k_rec with its slot sizes and record orders,
    k_short) produces the reference's bytes, on node-step records, '=' / 'X' CIGARs, interval steps with
    5-6 digit numbers and '*' lines."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    big = {"node_len_lo": 2000, "node_len_hi": 300000, "mrun_lo": 500, "mrun_hi": 150000, "steps_lo": 1, "steps_hi": 3, "max_runs": 4}
    for name, count, over in [("short", 40000, {"pct_star": 2}), ("short_eqx", 20000, {}), ("stable", 6000, big), ("short", 6000, big)]:
        p = H.preset(name, seed=77, **over)
        lengths = H.gen_lengths(p)
        gaf = H.gen_records(p, 0, count)
        cv = g2p.Converter(0)
        try:
            assert cv.load_lengths(lengths)
            out, res = cv.convert_host(gaf)
        finally:
            cv.close()
        rc, ref, err, kind = H.run_gaf2paf_cpu(gaf, lengths)
        assert rc == 0 and g2p.exit_code(res) == 0 and out == ref, (env, name)
        if env.get("G2P_FUSE") == "0":
            assert res.n_fused == 0
        elif env.get("G2P_FUSE") == "2" and name.startswith("short") and "node_len_lo" not in over:
            assert res.n_fused == res.n_records, "short canonical records are converted by k_fuse"


def test_mutation_fuzz_in_batches(g2p):
    """Mutated (malformed or unusual) records embedded in the middle of batches of valid short records,
    through the C-ABI in one process: stdout bytes, exit code and the exit(1) message must be the
    reference's, and the valid records before the bad one must come out (tests/fuzz_vs_ref.py's
    mutations; its per-process CLI form is the development tool)."""
    import random
    import fuzz_vs_ref as F
    rnd = random.Random(20261018)
    lengths = F.LENGTHS.encode()
    seeds = [s.replace(" ", "\t") for s in F.SEEDS]
    cv = g2p.Converter(0)
    bad = []
    try:
        assert cv.load_lengths(lengths)
        for case in range(300):
            line = F.mutate(rnd, rnd.choice(F.SEEDS))
            if rnd.random() < 0.3:
                line = F.mutate(rnd, line.replace("\t", " "))
            pre = [rnd.choice(seeds) for _ in range(rnd.randrange(0, 70))]
            post = [rnd.choice(seeds) for _ in range(rnd.randrange(0, 40))]
            gaf = ("\n".join(pre + [line] + post) + "\n").encode("latin-1")
            out, res = cv.convert_host(gaf)
            rc, ref_out, ref_err, kind = H.run_gaf2paf_cpu(gaf, lengths)
            if F.tolerated(line.encode("latin-1"), ref_out, out):
                continue
            ok = g2p.exit_code(res) == rc
            if rc == 134:
                ok = ok and ref_out.startswith(out) or (ok and out.startswith(ref_out))   # stdout is stdio-buffered when the reference aborts
            else:
                ok = ok and out == ref_out
            if rc == 1:
                ok = ok and g2p.Converter.format_error(res, gaf) == ref_err
            if not ok:
                bad.append((case, line, rc, g2p.exit_code(res)))
    finally:
        cv.close()
    assert not bad, bad[:5]
