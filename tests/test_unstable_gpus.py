"""gaf2unstable on several GPUs (G2P_GPUS=N): chunk s of the input goes to context s mod N, stdout, the multi-contig
warnings and the exit code stay those of one GPU and of the reference, and the rGFA tables are built once, on the
first context, and shared with the others (g2p_share_rgfa).

CPU: the executable's host logic (csrc/gaf2unstable_main.cpp, cli_pipeline.hpp) linked against the CPU stub of the
C-ABI (tests/hostsim/g2u_stub_capi.cpp: the library's table builder and the per-record code compiled for the host),
compared with the reference gaf2unstable (oracle/_ref, or the restatement when it is absent).
GPU (-m gpu): Converter.share_rgfa against the loading context, and bin/gaf2unstable with G2P_GPUS=2."""
import ctypes
import os
import subprocess
import tempfile

import pytest

import helpers as H

STUB = os.path.join(H.BUILD, "gaf2unstable_stub")
CHUNK = 6000                 # G2P_CHUNK_BYTES: ~45 chunks of the 3 000-record case, so chunks alternate contexts
BAD = b"q\t100\t0\t15\t+\t>nosuchcontig:0-15\t15\t0\t15\t15\t15\t60\tcg:Z:15M"   # unknown contig: the reference aborts


def stub():
    if not os.path.exists(STUB):
        subprocess.check_call(["make", "-C", H.ROOT, "build/gaf2unstable_stub"], stdout=subprocess.DEVNULL)
    return STUB


def run(binary, args, env=None, stdin=None, merged=False):
    """-> (exit code, stdout, stderr text); merged: stderr goes into the stdout pipe (their interleaving), stderr ''."""
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([binary] + args, input=stdin, stdout=subprocess.PIPE, stderr=subprocess.STDOUT if merged else subprocess.PIPE, env=e)
    rc = p.returncode if p.returncode >= 0 else 128 - p.returncode
    return rc, p.stdout, (p.stderr or b"").decode("latin-1")


def chunk_starts(gaf, chunk):
    """Byte offsets at which the executable's reader starts its chunks of a regular file (cli_pipeline.hpp)."""
    starts, pos = [], 0
    while pos < len(gaf):
        starts.append(pos)
        want = min(chunk, len(gaf) - pos)
        if pos + want >= len(gaf):
            break
        pos += gaf.rfind(b"\n", pos, pos + want) - pos + 1
    return starts


def chunk_of(starts, off):
    return max(i for i, s in enumerate(starts) if s <= off)


@pytest.fixture(scope="module")
def case():
    rgfa, gaf = H.gen_rgfa_case(41, n_records=3000, multi_ref_pct=6)
    with tempfile.TemporaryDirectory() as td:
        p = {k: os.path.join(td, k) for k in ("g.gfa", "a.gaf", "ref.tsv", "out.tsv")}
        open(p["g.gfa"], "wb").write(rgfa)
        open(p["a.gaf"], "wb").write(gaf)
        ref, _kind = H.oracle_path("auto", "gaf2unstable")
        r = run(ref, [p["a.gaf"], "-g", p["g.gfa"], "-o", p["ref.tsv"]])
        assert r[0] == 0
        yield p, rgfa, gaf, r, open(p["ref.tsv"], "rb").read()


@pytest.mark.parametrize("source", ["file", "stdin"])
@pytest.mark.parametrize("gpus", [1, 2, 3])
def test_matches_reference(case, gpus, source):
    p, rgfa, gaf, (rc0, out0, err0), nl0 = case
    assert len(chunk_starts(gaf, CHUNK)) > 6 * gpus
    assert err0.count("[gaf2unstable] warning") > 20
    env = {"G2P_GPUS": str(gpus), "G2P_CHUNK_BYTES": str(CHUNK)}
    if os.path.exists(p["out.tsv"]):
        os.remove(p["out.tsv"])
    if source == "file":
        r = run(stub(), [p["a.gaf"], "-g", p["g.gfa"], "-o", p["out.tsv"]], env)
    else:
        r = run(stub(), ["-", "-g", p["g.gfa"], "-o", p["out.tsv"]], env, stdin=gaf)
    assert r == (rc0, out0, err0)
    assert open(p["out.tsv"], "rb").read() == nl0


@pytest.mark.parametrize("gpus", [2, 3])
def test_warnings_interleave_with_stdout_as_on_one_gpu(case, gpus):
    """A chunk's warnings are printed before its output and after the previous chunk's, whichever context converted it:
    the merged stream equals the one-GPU stream, and each warning comes before the output line it quotes."""
    p, rgfa, gaf, (rc0, out0, err0), nl0 = case
    starts = chunk_starts(gaf, CHUNK)
    # the chunks that hold multi-contig records lie on every context
    warned = {chunk_of(starts, gaf.find(b"\n" + ln.split(b"\t", 1)[0] + b"\t") + 1)
              for ln in err0.encode("latin-1").split(b"\n") if ln.startswith(b"q")}
    assert {c % gpus for c in warned} == set(range(gpus))
    args = [p["a.gaf"], "-g", p["g.gfa"]]
    one = run(stub(), args, {"G2P_CHUNK_BYTES": str(CHUNK)}, merged=True)
    many = run(stub(), args, {"G2P_GPUS": str(gpus), "G2P_CHUNK_BYTES": str(CHUNK)}, merged=True)
    assert many == one and one[0] == 0
    merged, rest, pos = one[1], b"", 0
    while True:
        w = merged.find(b"[gaf2unstable] warning", pos)
        if w < 0:
            break
        a = merged.index(b"the (unstable) record is\n", w) + len(b"the (unstable) record is\n")
        b = merged.index(b"\n", a) + 1
        assert merged.find(b"\n" + merged[a:b], b - 1) >= 0, "a warning after the line it quotes"
        rest += merged[pos:w]
        pos = b
    assert rest + merged[pos:] == out0


def test_abort_in_a_chunk_of_the_second_context(case):
    """A record the reference aborts on, in a chunk that the second context converts: everything before it (output and
    warnings) is written, then SIGABRT (exit 134), identically on one and on two contexts."""
    p, rgfa, gaf, _r0, _nl0 = case
    starts = chunk_starts(gaf, CHUNK)
    c = next(i for i in range(len(starts) // 2, len(starts)) if i % 2 == 1)
    k = gaf.index(b"\n", starts[c] + 1) + 1          # the second line of chunk c
    bad = gaf[:k] + BAD + b"\n" + gaf[k:]
    assert chunk_of(chunk_starts(bad, CHUNK), k) == c
    ref, _kind = H.oracle_path("auto", "gaf2unstable")
    with tempfile.TemporaryDirectory() as td:
        bp = os.path.join(td, "bad.gaf")
        open(bp, "wb").write(bad)
        rrc, rout, rerr = run(ref, [bp, "-g", p["g.gfa"]])
        hrc, hout, herr = run(ref, ["-", "-g", p["g.gfa"]], stdin=gaf[:k])
        res = [run(stub(), [bp, "-g", p["g.gfa"]], {"G2P_GPUS": str(g), "G2P_CHUNK_BYTES": str(CHUNK)}) for g in (1, 2)]
    assert res[0] == res[1]
    rc, out, err = res[1]
    assert rrc == rc == 134 and hrc == 0
    assert out == hout and rout == out[:len(rout)]   # the reference may lose what is still in its stdio buffer
    assert err.startswith(herr) and herr.count("warning") > 0
    assert err[len(herr):].startswith("terminate: gaf2unstable cannot convert record 1 of this block") and err[len(herr):].count("\n") == 1


RGFA_FAIL = {
    # a rank-1 node between nodes of two reference contigs: rgfa-split's "Conflict found", exit 1
    "conflict": b"S\ts1\tACGT\tSN:Z:chr1\tSO:i:0\tSR:i:0\nS\ts2\tACGT\tSN:Z:chr2\tSO:i:0\tSR:i:0\nS\ts3\tAC\tSN:Z:alt\tSO:i:0\tSR:i:1\n"
                b"L\ts1\t+\ts3\t+\t0M\nL\ts3\t+\ts2\t+\t0M\n",
    # a rank-1 node without neighbours: "Unable to assign contigs", exit 1
    "unassigned": b"S\ts1\tACGT\tSN:Z:chr1\tSO:i:0\tSR:i:0\nS\ts3\tAC\tSN:Z:alt\tSO:i:0\tSR:i:1\n",
    # an S line without SO: assert, exit 134
    "no-so": b"S\ts1\tACGT\tSN:Z:chr1\tSR:i:0\n",
}


@pytest.mark.parametrize("name", sorted(RGFA_FAIL))
def test_rgfa_failures_are_the_same_on_two_contexts(case, name):
    p, rgfa, gaf, _r0, _nl0 = case
    ref, kind = H.oracle_path("auto", "gaf2unstable")
    with tempfile.TemporaryDirectory() as td:
        gp, lp = os.path.join(td, "bad.gfa"), os.path.join(td, "l.tsv")
        open(gp, "wb").write(RGFA_FAIL[name])
        rrc, rout, rerr = run(ref, [p["a.gaf"], "-g", gp])
        res = []
        for g in (1, 2):
            r = run(stub(), [p["a.gaf"], "-g", gp, "-o", lp], {"G2P_GPUS": str(g), "G2P_CHUNK_BYTES": str(CHUNK)})
            res.append(r + (os.path.exists(lp),))
    assert res[0] == res[1]
    rc, out, err, wrote = res[1]
    assert rc == rrc == (134 if name == "no-so" else 1)
    assert out == rout == b"" and not wrote
    if rc == 1:
        assert err == rerr


def test_stats_line_reports_the_gpus(case):
    p, rgfa, gaf, (rc0, out0, err0), nl0 = case
    rc, out, err = run(stub(), [p["a.gaf"], "-g", p["g.gfa"]], {"G2P_GPUS": "2", "G2P_CHUNK_BYTES": str(CHUNK), "G2P_STATS": "1"})
    assert rc == 0 and out == out0
    stats = [ln for ln in err.split("\n") if ln.startswith("[gaf2unstable] stats:")]
    assert stats[0] == "[gaf2unstable] stats: contexts ready"
    assert "records=%d " % gaf.count(b"\n") in stats[1] and " gpus=2 " in stats[1] and " rgfa=" in stats[1] and " share=" in stats[1]
    assert [ln for ln in err.split("\n") if not ln.startswith("[gaf2unstable] stats:")] == err0.split("\n")


# ---- GPU -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_share_rgfa_gives_the_loading_contexts_results(g2p):
    """A second context on the same GPU, given the tables with share_rgfa, converts like the context that loaded them,
    also after that one is destroyed."""
    rgfa, gaf = H.gen_rgfa_case(43, n_records=6000, aligned=True, multi_ref_pct=5)
    rc, ref, err, nl = H.run_gaf2unstable_ref(gaf, rgfa, True)
    assert rc == 0 and err
    bad = gaf + BAD + b"\n" + gaf[:3000]
    a, b, c, d = (g2p.Converter(0) for _ in range(4))
    try:
        vp = ctypes.c_void_p
        assert g2p.lib.g2p_share_rgfa(b._h, a._h) == g2p.G2P_E_NOTABLE      # nothing loaded yet
        assert g2p.lib.g2p_share_rgfa(a._h, a._h) == g2p.G2P_E_ARG
        assert g2p.lib.g2p_share_rgfa(None, a._h) == g2p.G2P_E_ARG and g2p.lib.g2p_share_rgfa(a._h, None) == g2p.G2P_E_ARG
        with pytest.raises(g2p.G2PError):
            b.share_rgfa(a)
        ok, code, msg = d.load_rgfa(RGFA_FAIL["conflict"])                  # a failed load leaves nothing to share
        assert not ok and code == 1
        assert g2p.lib.g2p_share_rgfa(c._h, d._h) == g2p.G2P_E_NOTABLE
        ok, code, msg = a.load_rgfa(rgfa)
        assert ok
        b.share_rgfa(a)
        assert b.node_lengths() == a.node_lengths() == nl
        ua = a.unstable_host(gaf)
        ub = b.unstable_host(gaf)
        assert ub[0] == ua[0] == ref and ub[2] == ua[2] and "".join(ub[2]) == err
        pa, ra, wa = a.unstable_convert_host(gaf)
        pb, rb, wb = b.unstable_convert_host(gaf)
        assert pb == pa and wb == wa == err and g2p.exit_code(rb) == g2p.exit_code(ra) == 0
        assert pb == H.run_gaf2paf_cpu(ref, nl)[1]
        xa, xb = a.unstable_host(bad), b.unstable_host(bad)
        assert xb[0] == xa[0] == ref and g2p.exit_code(xb[1]) == 134 and xb[1].err_record == xa[1].err_record == gaf.count(b"\n")
        a.close()
        c.share_rgfa(b)                                                     # the tables outlive the context that built them
        assert c.node_lengths() == nl
        out, res, warns = c.unstable_host(gaf)
        assert out == ref and "".join(warns) == err
    finally:
        for cv in (a, b, c, d):
            cv.close()


def n_gpus():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout
        return sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.gpu
def test_cli_on_two_gpus_matches_one_gpu_and_the_reference(g2p):
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    exe = os.path.join(g2p.BIN_DIR, "gaf2unstable")
    ref_exe, _kind = H.oracle_path("auto", "gaf2unstable")
    rgfa, base = H.gen_rgfa_case(45, n_records=50000, multi_ref_pct=2)
    gaf = base * 20                                                          # ~10^6 records
    env = {"G2P_CHUNK_MB": "4"}
    with tempfile.TemporaryDirectory() as td:
        gp, ap, bp = (os.path.join(td, x) for x in ("g.gfa", "a.gaf", "bad.gaf"))
        open(gp, "wb").write(rgfa)
        open(ap, "wb").write(gaf)
        lp = {g: os.path.join(td, "l%d.tsv" % g) for g in (0, 1, 2)}
        r0 = run(ref_exe, [ap, "-g", gp, "-o", lp[0]])
        r = {g: run(exe, [ap, "-g", gp, "-o", lp[g]], dict(env, G2P_GPUS=str(g))) for g in (1, 2)}
        assert r0[0] == 0 and r[1] == r[2] == r0
        assert open(lp[1], "rb").read() == open(lp[2], "rb").read() == open(lp[0], "rb").read()
        # stdin
        assert run(exe, ["-", "-g", gp], dict(env, G2P_GPUS="2"), stdin=gaf)[:2] == r0[:2]
        # a record the reference aborts on, in the second GPU's chunk (chunk 3 of 4 MB chunks)
        k = gaf.index(b"\n", 3 * (4 << 20) + 1000) + 1
        bad = gaf[:k] + BAD + b"\n" + gaf[k:]
        open(bp, "wb").write(bad)
        h = run(ref_exe, ["-", "-g", gp], stdin=gaf[:k])
        x = {g: run(exe, [bp, "-g", gp], dict(env, G2P_GPUS=str(g))) for g in (1, 2)}
        assert x[1] == x[2] and x[2][0] == 134 and h[0] == 0
        assert x[2][1] == h[1] and x[2][2].startswith(h[2]) and "terminate: gaf2unstable cannot convert" in x[2][2][len(h[2]):]
