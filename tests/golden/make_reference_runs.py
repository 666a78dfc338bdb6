#!/usr/bin/env python3
"""Generate tests/golden/reference_runs.json: what the reference executables print for the command lines that the tests
compare with them, so that those tests also run where the reference build (oracle/_ref) is absent.

    python tests/golden/make_reference_runs.py                   (after `make` and oracle/build_ref.sh)
    python tests/golden/make_reference_runs.py --source project  (without oracle/_ref: see below)

* "cli": argument errors of gaf2paf, gaffilter and gaf2unstable -- exit code, stdout and stderr, the program's own path
  written X and the paths of input files as the placeholders the arguments use ({L} lengths, {A} GAF, {G} graph).
* "gaffilter": gaffilter on the inputs of tests/test_filter.py's GPU tests (tests/helpers.py gen_filter_case) -- exit
  code, md5 and size of stdout (megabytes: too large to store), stderr.
* "gaffilter_inputs": every run of tests/test_filter.py's emulator tests (ref_gaffilter), keyed by the md5 of the input
  and the arguments -- exit code, md5 of stdout, last stderr line.

--source reference (the default) runs oracle/_ref/<tool> and stops when that build is missing.  --source project
records this project's executables and its filter kernels under the SIMT emulator (build/g2p_filter_simt) instead:
the tests then check that the project still does what it did when recorded, not what the reference does, so use it
only for outputs the same tests have already matched against the reference.  "source" in the file says which it was."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers as H  # noqa: E402

OUT = os.path.join(HERE, "reference_runs.json")

CLI = {
    "gaf2paf": [[], ["-l", "{L}"], ["{A}"], ["-h", "x"], ["-l", "/nonexistent/l.tsv", "{A}"], ["--bogus"],
                ["x.gaf"], ["-l", "/nonexistent/l.tsv", "x.gaf"], ["-h"], ["-l"], ["--lengths"], ["-z", "a"]],
    "gaffilter": [[], ["{A}"], ["-r", "2"], ["-r", "2", "/nonexistent.gaf"], ["--bogus"]],
    "gaf2unstable": [[], ["{A}"], ["{A}", "b", "c", "-g", "{G}"]],
}

# (gen_filter_case arguments, gaffilter arguments); "{A}" is the input as a file, "-" on stdin
FILTER = []
for paf in (False, True):
    p = ["-p"] if paf else []
    FILTER += [((21, 60000, 4000, paf), ["-r", "2"] + p + ["-"]),
               ((21, 60000, 4000, paf), ["-r", "5", "-m", "0.25", "-q", "5"] + p + ["-"]),
               ((21, 60000, 4000, paf), ["-o", "150", "-b", "60"] + p + ["-"])]
FILTER += [((31, 20000, 900, False), ["-r", "2", "{A}"]),
           ((31, 20000, 900, False), ["{A}", "-r", "5", "-m", "0.25"]),
           ((31, 20000, 900, False), ["-o", "100", "-"])]


def expand(args, subst):
    return [subst.get(a, a) for a in args]


def cli_runs(td, source):
    subst = {"{L}": os.path.join(td, "l.tsv"), "{A}": os.path.join(td, "a.gaf"), "{G}": os.path.join(td, "g.gfa")}
    rgfa, gaf = H.gen_rgfa_case(21, n_records=50, aligned=True)
    open(subst["{L}"], "wb").write(H.gen_lengths(H.preset("short", seed=77)))
    open(subst["{A}"], "wb").write(gaf)
    open(subst["{G}"], "wb").write(rgfa)
    own = {"gaf2paf": os.path.join(ROOT, "cactus-gfa-tools_b200", "bin", "gaf2paf"),
           "gaffilter": os.path.join(ROOT, "cactus-gfa-tools_b200", "bin", "gaffilter"),
           "gaf2unstable": os.path.join(ROOT, "cactus-gfa-tools_b200", "bin", "gaf2unstable")}
    runs = {}
    for tool, cases in CLI.items():
        exe = os.path.join(H.REF_BIN, tool) if source == "reference" else own[tool]
        runs[tool] = []
        for args in cases:
            rc, out, err = H.run_tool(exe, expand(args, subst), b"")
            assert "CUDA" not in err, (tool, args, err)   # argument handling ends before any device is opened
            err = err.replace(exe, "X")
            for k, v in subst.items():
                err = err.replace(v, k)
            runs[tool].append({"args": args, "rc": rc, "out": out.decode("latin-1"), "err": err})
    return runs


def filter_runs(td, source):
    ref = os.path.join(H.REF_BIN, "gaffilter")
    simt = os.path.join(H.BUILD, "g2p_filter_simt")
    runs = []
    for case, args in FILTER:
        text, _ = H.gen_filter_case(case[0], n_records=case[1], n_queries=case[2], paf=case[3])
        if source == "reference":
            path = os.path.join(td, "in.gaf")
            open(path, "wb").write(text)
            rc, out, err = H.run_tool(ref, expand(args, {"{A}": path}), text)
        else:   # the emulator reads stdin only
            rc, out, err = H.run_tool(simt, [a for a in args if a not in ("{A}", "-")] + ["-"], text)
        runs.append({"case": list(case), "args": args, "rc": rc, "md5": hashlib.md5(out).hexdigest(), "bytes": len(out), "err": err})
    return runs


def emulator_test_runs(source):
    """Run tests/test_filter.py's emulator tests with ref_gaffilter recording what it compares with."""
    with tempfile.TemporaryDirectory() as td:
        rec = os.path.join(td, "runs.jsonl")
        env = dict(os.environ, G2P_RECORD_GAFFILTER=rec)
        subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "not gpu", "-k", "emulated",
                               os.path.join(ROOT, "tests", "test_filter.py")], env=env, cwd=ROOT)
        runs = {}
        for line in open(rec):
            r = json.loads(line)
            runs[r.pop("key")] = r
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["reference", "project"], default="reference")
    a = ap.parse_args()
    if a.source == "reference":
        missing = [t for t in ("gaf2paf", "gaffilter", "gaf2unstable") if not os.path.exists(os.path.join(H.REF_BIN, t))]
        if missing:
            sys.exit("oracle/_ref/%s missing: run oracle/build_ref.sh first (or see --source)" % ", ".join(missing))
    if a.source == "project" and os.path.exists(os.path.join(H.REF_BIN, "gaffilter")):
        sys.exit("oracle/_ref is present: record from it (--source reference)")
    with tempfile.TemporaryDirectory() as td:
        d = {"note": "generated by tests/golden/make_reference_runs.py --source %s" % a.source,
             "source": a.source, "cli": cli_runs(td, a.source), "gaffilter": filter_runs(td, a.source)}
    d["gaffilter_inputs"] = emulator_test_runs(a.source)
    with open(OUT, "w") as f:
        json.dump(d, f, indent=1)
        f.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
