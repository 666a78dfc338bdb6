"""CPU tests: the oracle restatement (and the host instantiation of the device code)
against the committed golden vectors and, where the reference build is present,
against the reference binary on seeded synthetic inputs."""
import os
import subprocess
import tempfile

import pytest

import helpers as H

PORT = os.path.join(H.ORACLE_BIN, "gaf2paf_oracle")
HOSTSIM = os.path.join(H.BUILD, "g2p_hostsim")
SIMT = os.path.join(H.BUILD, "g2p_simt")   # the CUDA kernels themselves, run by the SIMT emulator (tests/hostsim/cuda_shim.hpp)
REF = os.path.join(H.REF_BIN, "gaf2paf")


def _run_vectors(binary):
    d = H.golden("gaf2paf_kat.json")
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "w").write(d["lengths"])
        for v in d["vectors"]:
            rc, out, err = H.run_tool(binary, ["-", "-l", lp], (v["in"] + "\n").encode("latin-1"))
            assert rc == v["rc"], v["name"]
            if rc != 134:
                assert out.decode("latin-1") == v["out"], v["name"]
            if rc == 1:
                assert err == v["err"], v["name"]
        rc, out, err = H.run_tool(binary, ["-", "-l", lp], ("\n".join(d["stream"]["in"]) + "\n").encode("latin-1"))
        assert rc == 0 and out.decode("latin-1") == d["stream"]["out"]


def test_oracle_port_matches_golden():
    _run_vectors(PORT)


def test_device_code_on_host_matches_golden():
    _run_vectors(HOSTSIM)


def test_kernels_under_simt_emulator_match_golden():
    """k_short / k_long / k_convert_list / scans / index kernels, executed warp-accurately on the CPU."""
    _run_vectors(SIMT)
    _run_vectors(SIMT + "_long")   # variant built with the k_short length limit at 0: every record goes through k_long


@pytest.mark.skipif(not os.path.exists(REF), reason="reference build (oracle/_ref) not present")
def test_reference_binary_matches_golden():
    _run_vectors(REF)


@pytest.mark.parametrize("name,count,over", [
    ("short", 3000, {"pct_star": 3}),
    ("short_eqx", 2000, {}),
    ("stable", 300, {}),
    ("medium", 300, {}),
    ("asm", 2, {"steps_lo": 800, "steps_hi": 1500}),
    # short records with 4..6-digit numbers (k_rec's loop paths) and with many tiny steps / ops
    ("short", 1500, {"node_len_lo": 2000, "node_len_hi": 300000, "mrun_lo": 500, "mrun_hi": 150000, "steps_lo": 1, "steps_hi": 3, "max_runs": 4}),
    ("stable", 1500, {"node_len_lo": 2000, "node_len_hi": 300000, "mrun_lo": 500, "mrun_hi": 150000, "steps_lo": 1, "steps_hi": 3, "max_runs": 4}),
    ("short_eqx", 1500, {"node_len_lo": 5, "node_len_hi": 40, "mrun_lo": 1, "mrun_hi": 12, "steps_lo": 1, "steps_hi": 7, "max_runs": 12, "indel_lo": 1, "indel_hi": 3}),
])
def test_differential_synthetic(name, count, over):
    """port == hostsim (== reference when built) on seeded synthetic records."""
    p = H.preset(name, seed=11, **over)
    lengths = H.gen_lengths(p)
    gaf = H.gen_records(p, 0, count, threads=4)
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "wb").write(lengths)
        rc_p, out_p, _ = H.run_tool(PORT, ["-", "-l", lp], gaf)
        rc_h, out_h, _ = H.run_tool(HOSTSIM, ["-", "-l", lp], gaf)
        assert rc_p == 0 and rc_h == 0
        assert out_p == out_h
        rc_s, out_s, _ = H.run_tool(SIMT, ["-", "-l", lp], gaf)
        assert rc_s == 0 and out_s == out_p
        assert out_p.count(b"\n") > 0
        if os.path.exists(REF):
            rc_r, out_r, _ = H.run_tool(REF, ["-", "-l", lp], gaf)
            assert rc_r == 0 and out_r == out_p


def test_unterminated_last_line_and_two_files():
    d = H.golden("gaf2paf_kat.json")
    lines = d["stream"]["in"]
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "w").write(d["lengths"])
        a, b = os.path.join(td, "a.gaf"), os.path.join(td, "b.gaf")
        half = len(lines) // 2
        open(a, "w").write("\n".join(lines[:half]))          # no trailing newline
        open(b, "w").write("\n".join(lines[half:]) + "\n")
        for binary in (PORT, HOSTSIM):
            rc, out, err = H.run_tool(binary, [a, b, "-l", lp])
            assert rc == 0 and out.decode("latin-1") == d["stream"]["out"], binary


# ---- gaf2unstable (config 2) ---------------------------------------------------------------
G2U_HOSTSIM = os.path.join(H.BUILD, "g2u_hostsim")
G2U_SIMT = os.path.join(H.BUILD, "g2u_simt")   # k_unstable<> (G2U_SIMT_STAGED=1: k_unstable_staged<>) under the SIMT emulator
G2U_PORT = os.path.join(H.ORACLE_BIN, "gaf2unstable_oracle")
# the kernels under the emulator: k_unstable, the library's default, over a grid of 3 CTAs (several stride turns), also
# with the CTAs in reverse order (the warning list fills in another order); k_unstable_staged; the staged kernel with
# tiny staging buffers (_small), so that some CTAs read / write global memory directly
G2U_SIMT_RUNS = {
    "list": (G2U_SIMT, {}),
    "list-reverse": (G2U_SIMT, {"G2P_SIMT_REVERSE": "1"}),
    "staged": (G2U_SIMT, {"G2U_SIMT_STAGED": "1"}),
    "staged-small": (G2U_SIMT + "_small", {}),
}


def run_g2u(binary, args, stdin, env=None):
    """-> (exit code, stdout, stderr text) of a gaf2unstable stand-in with `env` added to the environment."""
    p = subprocess.run([binary] + args, input=stdin, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=dict(os.environ, **(env or {})))
    return (p.returncode if p.returncode >= 0 else 128 - p.returncode), p.stdout, p.stderr.decode("latin-1")


@pytest.mark.parametrize("run", ["hostsim", "port"] + sorted(G2U_SIMT_RUNS))
def test_gaf2unstable_host_code_matches_golden(run):
    """the device code on the host, and the independent oracle restatement, against the golden vectors"""
    binary, env = {"hostsim": (G2U_HOSTSIM, {}), "port": (G2U_PORT, {})}.get(run) or G2U_SIMT_RUNS[run]
    d = H.golden("gaf2unstable_kat.json")
    with tempfile.TemporaryDirectory() as td:
        gp, lp = os.path.join(td, "g.gfa"), os.path.join(td, "nl.tsv")
        open(gp, "w").write(d["rgfa"])
        for v in d["vectors"]:
            rc, out, err = run_g2u(binary, ["-g", gp, "-"], (v["in"] + "\n").encode(), env)
            assert rc == v["rc"] and out.decode() == v["out"], v["in"]
        rc, out, err = run_g2u(binary, ["-g", gp, "-o", lp, "-"], ("\n".join(d["stream"]["in"]) + "\n").encode(), env)
        assert rc == 0 and out.decode() == d["stream"]["out"]
        assert open(lp).read() == d["node_lengths"]


@pytest.mark.parametrize("seed,aligned", [(1, False), (2, True), (3, False)])
def test_gaf2unstable_differential(seed, aligned):
    """device code on the host == reference binary (the restatement where the reference build is absent) on a synthetic
    rGFA + stable GAF, incl. the -o file."""
    rgfa, gaf = H.gen_rgfa_case(seed, n_records=600, aligned=aligned)
    rc, ref, err, nl = H.run_gaf2unstable_ref(gaf, rgfa, True)
    assert rc == 0
    assert err.count("[gaf2unstable] warning") > 3
    with tempfile.TemporaryDirectory() as td:
        gp, lp = os.path.join(td, "g.gfa"), os.path.join(td, "nl.tsv")
        open(gp, "wb").write(rgfa)
        for name, (binary, env) in [("hostsim", (G2U_HOSTSIM, {}))] + sorted(G2U_SIMT_RUNS.items()):
            rc, out, serr = run_g2u(binary, ["-g", gp, "-o", lp, "-"], gaf, env)
            assert rc == 0 and out == ref and open(lp, "rb").read() == nl, name
            assert serr == err, name   # the warnings verbatim and in record order
        rc, out, serr = H.run_tool(G2U_PORT, ["-g", gp, "-o", lp, "-"], gaf)   # oracle restatement: stderr verbatim too
        assert rc == 0 and out == ref and open(lp, "rb").read() == nl and serr == err


# ---- records delegated late (after k_long has already described some of their lines) ---------
def _late_cases():
    import re
    pm, ps = H.preset("medium", seed=5), H.preset("short", seed=5)
    lengths = H.gen_lengths(ps)
    med = H.gen_records(pm, 0, 6, threads=1).split(b"\n")[:-1]
    short = H.gen_records(ps, 0, 400, threads=1).split(b"\n")[:-1]

    def last_op(line, f):
        i = line.rfind(b"cg:Z:")
        j = line.find(b"\t", i)
        cg = line[i: j if j > 0 else len(line)]
        ops = re.findall(rb"\d+[A-Z=]", cg[5:])
        ops[-1] = f(ops[-1])
        return line[:i] + b"cg:Z:" + b"".join(ops) + (line[j:] if j > 0 else b"")

    noncanon = last_op(med[4], lambda o: b"0" + o)        # leading zero in the last op: valid, not canonical
    abort = last_op(med[2], lambda o: o[:-1] + b"Q")      # invalid letter at the very end: the reference aborts
    return lengths, {
        "late-noncanonical": med[:2] + short[:150] + [noncanon] + short[150:300] + [med[5]] + short[300:],
        "late-abort-last": med[:2] + short[:150] + [noncanon] + short[150:] + [abort],
        "late-abort-middle": med[:2] + short[:150] + [abort] + short[150:],
    }


@pytest.mark.parametrize("reverse", [False, True])
def test_late_delegation_under_emulator(reverse):
    """k_long describes a long record batch by batch; when the record turns out non-canonical near
    its end it is delegated, and the lines already described must not be emitted from the
    descriptors.  Run with the emulator's CTAs in both orders."""
    ref_bin, _kind = H.oracle_path()   # the reference build when present, else the restatement
    lengths, cases = _late_cases()
    env = dict(os.environ, G2P_SIMT_REVERSE="1") if reverse else dict(os.environ)
    import subprocess
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "wb").write(lengths)
        for name, lines in cases.items():
            data = b"\n".join(lines) + b"\n"
            rc, ref, err = H.run_tool(ref_bin, ["-", "-l", lp], data)
            for binary in (SIMT, SIMT + "_long"):
                p = subprocess.run([binary, "-l", lp, "-"], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
                got_rc = p.returncode if p.returncode >= 0 else 128 - p.returncode
                assert got_rc == rc, name
                assert (p.stdout == ref) if rc != 134 else ref.startswith(p.stdout), name


def test_gaf2unstable_many_tags():
    """Optional fields: none, more than the 16 the per-record code collects (it rescans the text then), duplicates before
    and after that limit, long names, an rc tag that is replaced -- each record alone, stdout / exit code as the reference
    (the restatement where the reference build is absent)."""
    ref_bin, _kind = H.oracle_path("auto", "gaf2unstable")
    rgfa, gaf = H.gen_rgfa_case(4, n_records=40, aligned=True)
    base = [l for l in gaf.split(b"\n") if l and not l.startswith(b"*") and l.split(b"\t")[5] != b"*"][:6]
    assert len(base) >= 4

    def with_tags(line, tags):
        return b"\t".join(line.split(b"\t")[:12] + tags)
    many = [("%c%c:i:%d" % (97 + i // 5, 97 + i % 5, i)).encode() for i in range(22)]
    cases = [
        with_tags(base[0], []),
        with_tags(base[1], many[:16][::-1]),
        with_tags(base[2], many[:17][::-1]),
        with_tags(base[3], many[::-1] + [b"rc:Z:old", b"longname:Z:x", b"lo:Z:y"]),
        with_tags(base[0], many[:10] + [many[3]]),                    # duplicate among the collected fields
        with_tags(base[1], many[:20] + [many[2]]),                    # duplicate of a collected field after the limit
        with_tags(base[2], many[:20] + [many[18]]),                   # duplicate of a field beyond the limit
        with_tags(base[3], [b"ab:i:1", b"abc:i:2", b"a:i:3x", b"ab:Z:dup"]),
        with_tags(base[0], [b"zz:i:1", b"", b"aa:i:2", b""]),           # empty fields
        with_tags(base[1], [b"bad"]),
    ]
    with tempfile.TemporaryDirectory() as td:
        gp = os.path.join(td, "g.gfa")
        open(gp, "wb").write(rgfa)
        for c in cases:
            data = base[4] + b"\n" + c + b"\n" + base[5] + b"\n"
            rc, ref, err = H.run_tool(ref_bin, ["-g", gp, "-"], data)
            runs = [(G2U_HOSTSIM, {})] + list(G2U_SIMT_RUNS.values()) + ([(G2U_PORT, {})] if ref_bin != G2U_PORT else [])
            for binary, env in runs:
                rc1, out1, _ = run_g2u(binary, ["-g", gp, "-"], data, env)
                assert rc1 == rc, (binary, env, c)
                assert (out1 == ref) if rc == 0 else ref.startswith(out1) or out1.startswith(ref), (binary, env, c)
