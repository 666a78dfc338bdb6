#!/usr/bin/env python3
"""gaf2unstable on several GPUs: wall time of bin/gaf2unstable, file -> /dev/null, with G2P_GPUS = 1, 2, 4, 8 (the counts
this box has; the others are reported as not measured).  Each count runs --repeat times; the G2P_STATS line gives the
time of the pipeline (after the contexts exist and the tables are on every GPU), the rGFA load on the first context
(host build + upload) and the copy of the tables to the other GPUs, reported separately.  One more run per count
hashes stdout, which must be the same for every count.  The input is K copies of a seeded gen_rgfa_case of 10 000
records on a 500-contig rGFA, written to a temporary file.  The card's name and power limit are read in the same run.

    python tools/unstable_scale.py [--records 10000000] [--gpus 1,2,4,8] [--repeat 3] [--out profiles/r04_unstable_scale.txt]"""
import argparse, hashlib, json, os, re, shutil, statistics, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import cactus_gfa_tools_b200 as g2p, helpers as H

ap = argparse.ArgumentParser()
ap.add_argument("--records", type=int, default=10_000_000)
ap.add_argument("--gpus", default="1,2,4,8")
ap.add_argument("--repeat", type=int, default=3)
ap.add_argument("--out", default=None)
a = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
have = len(smi)
if have == 0:
    sys.exit("unstable_scale: no GPU")
rgfa, base = H.gen_rgfa_case(71, n_contigs=500, n_records=10000, multi_ref_pct=1)
n_base = base.count(b"\n")
copies = -(-a.records // n_base)
exe = os.path.join(g2p.BIN_DIR, "gaf2unstable")
STATS = re.compile(r"stats: records=(\d+) in=(\d+) B out=(\d+) B device=([\d.]+) ms wall=([\d.]+) s gpus=(\d+) rgfa=([\d.]+) s share=([\d.]+) s")

td = tempfile.mkdtemp()
rows = []
try:
    gp, path, errp = (os.path.join(td, x) for x in ("g.gfa", "in.gaf", "err.txt"))
    open(gp, "wb").write(rgfa)
    if shutil.disk_usage(td).free < len(base) * copies + (1 << 30):
        sys.exit("unstable_scale: %s has less than %d bytes free" % (td, len(base) * copies))
    with open(path, "wb") as f:
        for _ in range(copies):
            f.write(base)
    size = os.path.getsize(path)

    def run(g, stdout):
        env = dict(os.environ, G2P_GPUS=str(g), G2P_STATS="1")
        with open(errp, "wb") as ef:
            t0 = time.perf_counter()
            p = subprocess.Popen([exe, path, "-g", gp], stdout=stdout, stderr=ef, env=env)
            h = hashlib.md5()
            if stdout == subprocess.PIPE:
                for blk in iter(lambda: p.stdout.read(1 << 24), b""):
                    h.update(blk)
            rc = p.wait()
            wall = time.perf_counter() - t0
        with open(errp, "rb") as ef:
            ef.seek(max(0, os.path.getsize(errp) - 4096))
            tail = ef.read().decode("latin-1")
        assert rc == 0, tail
        m = STATS.findall(tail)[-1]
        return wall, m, h.hexdigest()

    md5 = {}
    for g in [int(x) for x in a.gpus.split(",")]:
        if g > have:
            rows.append(dict(gpus=g, result="not measured: this box has %d GPU%s" % (have, "" if have == 1 else "s")))
            print(json.dumps(rows[-1]), flush=True)
            continue
        runs = [run(g, subprocess.DEVNULL) for _ in range(a.repeat)]
        md5[g] = run(g, subprocess.PIPE)[2]
        pipe = [float(m[4]) for _, m, _ in runs]
        m0 = runs[0][1]
        r = dict(gpus=g, records=int(m0[0]), in_bytes=int(m0[1]), out_bytes=int(m0[2]),
                 process_s=[round(w, 3) for w, _, _ in runs], pipeline_s=pipe, pipeline_median_s=statistics.median(pipe),
                 records_per_s=round(int(m0[0]) / statistics.median(pipe)), device_ms=[float(m[3]) for _, m, _ in runs],
                 rgfa_load_s=[float(m[6]) for _, m, _ in runs], rgfa_share_s=[float(m[7]) for _, m, _ in runs], stdout_md5=md5[g])
        rows.append(r)
        print(json.dumps(r), flush=True)
    assert len(set(md5.values())) <= 1, "stdout differs between GPU counts: %r" % md5
finally:
    shutil.rmtree(td, ignore_errors=True)

head = ("# tools/unstable_scale.py: bin/gaf2unstable file -> /dev/null, %d copies of gen_rgfa_case(71, n_contigs=500, n_records=10000, "
        "multi_ref_pct=1): %d records, %d B of GAF; rGFA %d B, %d S lines; %d runs per GPU count; cards: %s"
        % (copies, n_base * copies, size, len(rgfa), rgfa.count(b"\nS") + 1, a.repeat, "; ".join(smi)))
text = head + "\n" + "\n".join(json.dumps(r) for r in rows) + "\n"
print(text)
if a.out:
    with open(a.out, "w") as f:
        f.write(text)
