#!/usr/bin/env python3
"""gaffilter on multi-GB inputs: wall time of the gaffilter executable with G2P_GPUS = 1, 2, 4, 8 (the counts this box
has), with the filter job's per-pass device time and PCIe bytes (G2P_STATS=1), and a 3.5 GB input through the single
g2p_filter_host call for comparison.  The inputs are K renamed copies (query names prefixed c{k}_) of a gen_filter_case
base of 60 000 records, written to a temporary file.  The card's name and power limit are read in the same run.

    python tools/filter_scale.py [--gb 6] [--gpus 1,2,4,8] [--out profiles/r03_filter_scale.txt]"""
import argparse, json, os, re, shutil, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import cactus_gfa_tools_b200 as g2p, helpers as H

ap = argparse.ArgumentParser()
ap.add_argument("--gb", type=float, default=6.0, help="size of the job's input in GB (> 4.29 GB: beyond the single call)")
ap.add_argument("--single-gb", type=float, default=3.5)
ap.add_argument("--gpus", default="1,2,4,8")
ap.add_argument("--out", default=None)
a = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
have = len(smi)
base, _ = H.gen_filter_case(61, 60000, 4000, False)


def renamed(k):
    pre = b"c%d_" % k
    t = base.replace(b"\nq", b"\n" + pre + b"q")
    return pre + t if t.startswith(b"q") else t


exe = os.path.join(g2p.BIN_DIR, "gaffilter")
td = tempfile.mkdtemp()
rows = []
try:
    need = int(a.gb * 1e9) + (1 << 30)
    if shutil.disk_usage(td).free < need:
        sys.exit("filter_scale: %s has less than %d bytes free" % (td, need))
    path = os.path.join(td, "in.gaf")

    def run(env_extra, label, size):
        env = dict(os.environ, G2P_STATS="1", **env_extra)
        t0 = time.perf_counter()
        p = subprocess.run([exe, "-r", "2", path], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=env)
        wall = time.perf_counter() - t0
        err = p.stderr.decode()
        assert p.returncode == 0, err[-500:]
        r = dict(label=label, bytes=size, wall_s=round(wall, 3), summary=err.strip().split("\n")[-1 if "stats" not in err else -2])
        m = re.search(r"load=([\d.]+) ms decide=([\d.]+) ms emit=([\d.]+) ms h2d=(\d+) B d2h=(\d+) B", err)
        if m:
            r.update(load_ms=float(m.group(1)), decide_ms=float(m.group(2)), emit_ms=float(m.group(3)), h2d_bytes=int(m.group(4)), d2h_bytes=int(m.group(5)))
        rows.append(r)
        print(json.dumps(r), flush=True)

    k = 0
    with open(path, "wb") as f:
        while f.tell() + len(base) <= a.single_gb * 1e9:
            f.write(renamed(k)); k += 1
    size = os.path.getsize(path)
    run({}, "single call, 1 GPU", size)
    with open(path, "ab") as f:
        while f.tell() + len(base) <= a.gb * 1e9:
            f.write(renamed(k)); k += 1
    size = os.path.getsize(path)
    for g in [int(x) for x in a.gpus.split(",")]:
        if g > have:
            rows.append(dict(label="job, %d GPUs" % g, skipped="this box has %d GPUs" % have))
            print(json.dumps(rows[-1]), flush=True)
            continue
        run({"G2P_GPUS": str(g)}, "job, %d GPUs" % g, size)
finally:
    shutil.rmtree(td, ignore_errors=True)

head = "# tools/filter_scale.py: gaffilter -r 2 on K renamed copies of gen_filter_case(61, 60000, 4000); cards: %s" % "; ".join(smi)
text = head + "\n" + "\n".join(json.dumps(r) for r in rows) + "\n"
print(text)
if a.out:
    with open(a.out, "w") as f:
        f.write(text)
