"""Host logic of the gaf2paf executable on the CPU: csrc/gaf2paf_main.cpp (getopt table, the
reader -> per-GPU converter -> writer pipeline of cli_pipeline.hpp, chunk cutting, multi-file and stdin
input, G2P_GPUS round-robin with ordered output, error / exit-code paths) linked against a CPU stub of the
C-ABI (tests/hostsim/g2p_stub_capi.cpp -- the product's scalar device code compiled for the host), compared
byte for byte with the reference gaf2paf (oracle/_ref, or the restatement when it is absent).

The reference analogue is the in-order loop over the inputs, gaf2paf_main.cpp:342-374."""
import os
import subprocess
import tempfile

import pytest

import helpers as H

STUB = os.path.join(H.BUILD, "gaf2paf_stub")


def run(binary, args, env=None, stdin=None, stdout_path=None):
    e = dict(os.environ)
    e.update(env or {})
    if stdout_path:
        with open(stdout_path, "wb") as f:
            p = subprocess.run([binary] + args, input=stdin, stdout=f, stderr=subprocess.PIPE, env=e)
        out = open(stdout_path, "rb").read()
    else:
        p = subprocess.run([binary] + args, input=stdin, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e)
        out = p.stdout
    rc = p.returncode if p.returncode >= 0 else 128 - p.returncode
    return rc, out, p.stderr.decode("latin-1")


@pytest.fixture(scope="module")
def case():
    p = H.preset("short", seed=77, pct_star=1)
    pm = H.preset("medium", seed=77)
    lengths = H.gen_lengths(p)
    a = H.gen_records(p, 0, 3000, threads=2)
    b = H.gen_records(pm, 0, 30, threads=2) + H.gen_records(p, 3000, 1500, threads=2)
    with tempfile.TemporaryDirectory() as td:
        paths = {k: os.path.join(td, k) for k in ("l.tsv", "a.gaf", "b.gaf", "out.paf")}
        open(paths["l.tsv"], "wb").write(lengths)
        open(paths["a.gaf"], "wb").write(a)
        open(paths["b.gaf"], "wb").write(b[:-1])   # last line of the second file lacks its newline
        yield paths, a, b


@pytest.mark.parametrize("env", [
    {},
    {"G2P_CHUNK_BYTES": "5000"},
    {"G2P_CHUNK_BYTES": "20000", "G2P_GPUS": "3"},
    {"G2P_CHUNK_BYTES": "300", "G2P_GPUS": "2"},          # chunks shorter than some records: the reader keeps growing them
    {"G2P_CHUNK_BYTES": "70000", "G2P_IO_MIN_BYTES": "4096", "G2P_IO_THREADS": "4"},   # parallel pread
])
def test_two_files_match_reference(case, env):
    paths, a, b = case
    ref, _kind = H.oracle_path()
    args = ["-l", paths["l.tsv"], paths["a.gaf"], paths["b.gaf"]]
    rc0, out0, err0 = run(ref, args)
    rc1, out1, err1 = run(STUB, args, env)
    assert (rc1, err1) == (rc0, err0) == (0, "")
    assert out1 == out0


def test_stdout_regular_file_parallel_pwrite_and_stdin(case):
    paths, a, b = case
    ref, _kind = H.oracle_path()
    rc0, out0, _ = run(ref, ["-l", paths["l.tsv"], paths["a.gaf"], "-"], stdin=b)
    env = {"G2P_CHUNK_BYTES": "100000", "G2P_IO_MIN_BYTES": "8192", "G2P_IO_THREADS": "4", "G2P_GPUS": "2"}
    rc1, out1, err1 = run(STUB, ["-l", paths["l.tsv"], paths["a.gaf"], "-"], env, stdin=b, stdout_path=paths["out.paf"])
    assert rc0 == rc1 == 0 and err1 == ""
    assert out1 == out0
    # options after the positionals (GNU permute), like the reference
    rc2, out2, _ = run(STUB, [paths["a.gaf"], "-l", paths["l.tsv"]], {"G2P_CHUNK_BYTES": "9000"})
    rc3, out3, _ = run(ref, [paths["a.gaf"], "-l", paths["l.tsv"]])
    assert rc2 == rc3 == 0 and out2 == out3


@pytest.mark.parametrize("env", [{}, {"G2P_CHUNK_BYTES": "4000", "G2P_GPUS": "2"}])
@pytest.mark.parametrize("kind", ["name", "nocg", "abort"])
def test_error_in_a_later_chunk_stops_like_the_reference(case, env, kind):
    paths, a, b = case
    ref, _kind = H.oracle_path()
    lines = a.split(b"\n")
    k = 1700
    f = lines[k].split(b"\t")
    if kind == "name":
        f[5] = b">nosuchnode" + f[5]
    elif kind == "nocg":
        f = [x for x in f if not x.startswith(b"cg:Z:")]
    else:
        f[1] = b""
    lines[k] = b"\t".join(f)
    with tempfile.TemporaryDirectory() as td:
        gp = os.path.join(td, "bad.gaf")
        open(gp, "wb").write(b"\n".join(lines))
        args = ["-l", paths["l.tsv"], gp, paths["b.gaf"]]
        rc0, out0, err0 = run(ref, args)
        rc1, out1, err1 = run(STUB, args, env)
    assert rc1 == rc0 and rc0 in (1, 134)
    if rc0 == 1:
        assert err1 == err0 and out1 == out0
    else:
        # SIGABRT: the reference may lose stdout bytes still in its stdio buffer; what it did write is a prefix
        assert out1.startswith(out0) or out0.startswith(out1)


def test_missing_second_input_reports_after_the_first_is_written(case):
    paths, a, b = case
    ref, _kind = H.oracle_path()
    args = ["-l", paths["l.tsv"], paths["a.gaf"], "/nonexistent/x.gaf", paths["b.gaf"]]
    rc0, out0, err0 = run(ref, args)
    rc1, out1, err1 = run(STUB, args, {"G2P_CHUNK_BYTES": "50000", "G2P_GPUS": "2"})
    assert (rc1, out1, err1) == (rc0, out0, err0)
    assert rc0 == 1 and len(out0) > 0


def test_usage_errors_match(case):
    paths, a, b = case
    subst = {"{L}": paths["l.tsv"], "{A}": paths["a.gaf"]}
    for args in ([], ["-l", "{L}"], ["{A}"], ["-h", "x"], ["-l", "/nonexistent/l.tsv", "{A}"], ["--bogus"]):
        rc0, out0, err0 = H.reference_cli("gaf2paf", args, subst)
        rc1, out1, err1 = run(STUB, [subst.get(x, x) for x in args])
        assert rc1 == rc0 and out1 == out0
        assert err1.replace(STUB, "X") == err0
