#!/usr/bin/env python3
"""bench.py — gaf2paf throughput on B200 (BASELINE.json metric: GAF records/s and input GB/s
vs the HBM roofline), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload short|tagged|mixed|stable|medium|asm|unstable] [--records R]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's CPU gaf2paf on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's output to DIR/*.npy (see dump_outputs)

A step is one pass of the whole device pipeline (DESIGN.md §4) over one synthetic batch.  The inputs are generated
from fixed seeds, so runs with the same arguments convert the same bytes.

* `value`  — the batch already resident in HBM (CUDA events around exactly K steps, max over ranks).
* `e2e`    — the same metric through the host-buffer C-ABI call g2p_convert_host (pinned host input ->
             H2D -> pipeline -> D2H into pinned host memory), i.e. what the gaf2paf executable does per chunk.
* `cli`    — the drop-in executable itself: bin/gaf2paf file -> /dev/null (and file -> file) from tmpfs, one
             process driving all N GPUs (G2P_GPUS=N), wall clock; rank 0 runs it while the other ranks wait.

Multi-GPU (--gpus N, one process per GPU): ONE logical input — the concatenation of the ranks' generated
record ranges, written to a shared tmpfs file — is cut into N newline-aligned byte ranges
(cactus_gfa_tools_b200.shard_ranges, SURVEY.md §8e) and rank r converts range r; the per-shard outputs are in
record order when taken in rank order (no collective on the data path; NCCL only carries the timing barrier
and two small all-gathers of sizes).  Per-GPU work is fixed as N grows: "scaling": "weak".
"""
import argparse
import ctypes
import hashlib
import json
import mmap
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # BASELINE.json configs[2]: synthetic 10M-record short-read GAF on 1 B200
    "short": {"preset": "short", "records": 10_000_000, "desc": "configs[2]: synthetic short-read GAF, 1-5 node steps, short cg CIGARs",
              "cpu_records": 400_000},
    # short reads with instrument-style names and a long extra tag: 250-500 B records
    "tagged": {"preset": "tagged", "records": 5_000_000, "desc": "configs[2] variant: short-read records of 250-500 B (40 B read names, 120 B extra tag)",
               "cpu_records": 300_000},
    # BASELINE.json configs[4] shape at a size that fits the harness: ~90 % of the bytes short-read records,
    # ~10 % assembly-scale records (one every 16 400 records), one 2 M-node table
    "mixed": {"preset": "mixed", "records": 8_000_000, "desc": "configs[4] shape: mixed GAF, ~90 % of the bytes short-read records and ~10 % assembly-scale records (5k-15k steps), sharded by newline-aligned byte ranges",
              "cpu_records": 16_400 * 4},
    # shapes of configs[0] / configs[1] (stable-interval and node-coordinate assembly alignments)
    "stable": {"preset": "stable", "records": 300_000, "desc": "configs[0] shape: stable-interval steps (>contig:start-end), ~2 kB records", "cpu_records": 40_000},
    "medium": {"preset": "medium", "records": 100_000, "desc": "configs[1] shape: node-coordinate records of 20-200 steps, ~2 kB", "cpu_records": 6_000},
    # BASELINE.json configs[1]: gaf2unstable + gaf2paf on an rGFA, as ONE device-resident call (N2, SURVEY.md §8f)
    "unstable": {"kind": "unstable", "preset": None, "records": 300_000, "cpu_records": 100_000,
                 "desc": "configs[1] shape: gaf2unstable | gaf2paf fused (stable-interval GAF + rGFA -> node-space PAF, the intermediate GAF stays on the device)"},
    "asm": {"preset": "asm", "records": 4000, "desc": "configs[3] shape: assembly-scale records, 5k-15k steps, 4000 of the 100k records (PAF of all would not fit next to the input)",
            "cpu_records": 40},
}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def scratch_dir(need_bytes):
    """tmpfs when it has room (the inputs of both arms are read from memory, not from a disk), else the temp dir."""
    for d in ("/dev/shm", tempfile.gettempdir()):
        try:
            st = os.statvfs(d)
            if st.f_bavail * st.f_frsize > need_bytes * 1.2 + (256 << 20):
                return d
        except OSError:
            pass
    return tempfile.gettempdir()


class CpuArm:
    """The CPU gaf2paf (oracle/_ref reference build when present, else the restatement) on a bounded sample of
    the workload: `procs` independent processes on disjoint record ranges, inputs in tmpfs, stdout to /dev/null.
    The lengths-table load is timed separately (the binary on an empty GAF) and EXCLUDED from the rate, like the
    GPU arm's g2p_load_lengths, which runs before its timed region; both lines print `table_load_s`."""

    def __init__(self, H, preset_name, seed, per_proc, procs):
        self.binary, self.kind = H.oracle_path()
        self.per, self.procs = max(1, per_proc), procs
        self.td = tempfile.TemporaryDirectory(dir=scratch_dir(max(self.per * procs * 300, 1 << 30)))
        td = self.td.name
        self.lp = os.path.join(td, "l.tsv")
        self.empty = os.path.join(td, "empty.gaf")
        open(self.empty, "wb").close()
        self.files, self.nbytes = [], 0
        self.unstable = preset_name is None
        if self.unstable:
            # the reference's two-stage pipeline, stage after stage: gaf2unstable in.gaf -g g.gfa -o L > u.gaf; gaf2paf u.gaf -l L
            self.binary_u, _ = H.oracle_path("auto", "gaf2unstable")
            rgfa, gaf = H.gen_rgfa_case(seed, n_contigs=24, n_records=self.per, aligned=True)
            self.gp = os.path.join(td, "g.gfa")
            open(self.gp, "wb").write(rgfa)
            open(self.lp, "wb").close()
            for i in range(procs):
                fp = os.path.join(td, "s%d.gaf" % i)
                open(fp, "wb").write(gaf)
                self.files.append(fp)
                self.nbytes += len(gaf)
            self.per = gaf.count(b"\n")
            self.table_load_s = 0.0
            return
        p = H.preset(preset_name, seed=seed)
        open(self.lp, "wb").write(H.gen_lengths(p))
        for i in range(procs):
            g = H.gen_records(p, i * self.per, self.per)
            fp = os.path.join(td, "s%d.gaf" % i)
            open(fp, "wb").write(g)
            self.files.append(fp)
            self.nbytes += len(g)
        # table load + process start, all processes at once like the timed runs
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            ps = [subprocess.Popen([self.binary, self.empty, "-l", self.lp], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for _ in range(procs)]
            for q in ps:
                q.wait()
            ts.append(time.perf_counter() - t0)
        self.table_load_s = min(ts)

    def step(self):
        if self.unstable:
            t0 = time.perf_counter()
            cmd = '"%s" "$0" -g "%s" -o "$0.L" > "$0.u" 2>/dev/null && "%s" "$0.u" -l "$0.L" > /dev/null' % (self.binary_u, self.gp, self.binary)
            ps = [subprocess.Popen(["bash", "-c", cmd, fp]) for fp in self.files]
            rcs = [q.wait() for q in ps]
            dt = time.perf_counter() - t0
            if any(rcs):
                raise RuntimeError("cpu baseline (gaf2unstable | gaf2paf) failed: rc %r" % rcs)
            return dt
        t0 = time.perf_counter()
        ps = [subprocess.Popen([self.binary, fp, "-l", self.lp], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for fp in self.files]
        rcs = [q.wait() for q in ps]
        dt = time.perf_counter() - t0
        if any(rcs):
            raise RuntimeError("cpu baseline failed: rc %r" % rcs)
        return dt

    def result(self, dts):
        wall = sum(dts)
        conv = max(1e-9, wall - self.table_load_s * len(dts))
        n = self.per * self.procs * len(dts)
        return {"value": n / conv, "unit": "records/s", "cores": self.procs, "kind": self.kind,
                "sample": "%d records (%d B) of the same workload per step, %d process(es) x %d records, %d step(s); lengths-table load (%.3f s, timed on an empty GAF) excluded"
                          % (self.per * self.procs, self.nbytes, self.procs, self.per, len(dts), self.table_load_s),
                "seconds": wall, "table_load_s": self.table_load_s, "value_incl_table_load": n / wall,
                "input_MBps": self.nbytes * len(dts) / conv / 1e6}

    def close(self):
        self.td.cleanup()


DUMP_WINDOWS, DUMP_WINDOW_BYTES = 128, 64 << 10   # the output text sample: 8 MiB of bytes, 32 MiB as float32


def dump_outputs(dirname, g2p, d_out, res, suffix=""):
    """--dump-outputs: what the timed call returned in its last step, for comparing two builds output for output.

    paf.npy              the output text as byte values (float32): all of it when it fits the sample, else
                         DUMP_WINDOWS windows of DUMP_WINDOW_BYTES at offsets drawn with a fixed seed
    paf_offsets.npy      the start offset of each window (float64)
    paf_byte_counts.npy  how often each byte value 0..255 occurs in the whole output (float64)
    paf_md5.npy          the 16 bytes of the md5 digest of the whole output (float64): equal only for equal outputs
    result.npy           n_records, out_bytes, exit code, rec_status, rec_aux, err_record, stage, mid_bytes (float64);
                         timings and per-kernel record counts are left out, they are not part of the result"""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    n = int(res.out_bytes)
    if n <= DUMP_WINDOWS * DUMP_WINDOW_BYTES:
        offsets = np.zeros(1, dtype=np.int64)
        sample = np.frombuffer(g2p.copy_to_host(d_out, n), dtype=np.uint8)
    else:
        offsets = np.sort(np.random.default_rng(0).choice(n - DUMP_WINDOW_BYTES + 1, DUMP_WINDOWS, replace=False))
        sample = np.concatenate([np.frombuffer(g2p.copy_to_host(d_out + int(o), DUMP_WINDOW_BYTES), dtype=np.uint8) for o in offsets])
    counts = np.zeros(256, dtype=np.int64)
    digest = hashlib.md5()
    chunk = 64 << 20
    for o in range(0, n, chunk):
        part = g2p.copy_to_host(d_out + o, min(chunk, n - o))
        counts += np.bincount(np.frombuffer(part, dtype=np.uint8), minlength=256)
        digest.update(part)
    fields = [res.n_records, res.out_bytes, g2p.exit_code(res), res.rec_status, res.rec_aux, res.err_record, res.stage, res.mid_bytes]
    for name, arr in (("paf", sample.astype(np.float32)), ("paf_offsets", offsets.astype(np.float64)),
                      ("paf_byte_counts", counts.astype(np.float64)), ("paf_md5", np.frombuffer(digest.digest(), dtype=np.uint8).astype(np.float64)),
                      ("result", np.array(fields, dtype=np.float64))):
        np.save(os.path.join(dirname, name + suffix + ".npy"), arr)


def run_reference(a):
    """--impl reference: the reference's own CPU implementation on the host cores."""
    import helpers as H
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[a.workload]
    procs = min(os.cpu_count() or 1, 64)
    arm = CpuArm(H, wl["preset"], 1000 if wl["preset"] else 7, wl["cpu_records"], procs)
    try:
        dts = []
        for s in range(a.warmup + a.steps):
            dt = arm.step()
            if s >= a.warmup:
                dts.append(dt)
        r = arm.result(dts)
    finally:
        arm.close()
    line = {
        "impl": "reference", "metric": "gaf2paf_records_per_s", "value": r["value"], "unit": "records/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 * r["seconds"] / max(1, len(dts)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": wl["desc"], "preset": wl["preset"], "records_per_step": wl["cpu_records"] * procs,
                   "same_config": "same generator, preset and seed family as the GPU arm; a bounded sample per step (the full 10 M records take ~55 s per core), "
                                  "table load excluded from both arms"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "table_load_s": r["table_load_s"], "value_incl_table_load": r["value_incl_table_load"],
        "input_MBps": r["input_MBps"], "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_cli(g2p, gaf_path, lengths_path, n_gpus, n_records, in_bytes, out_dir):
    """bin/gaf2paf on the shared input file, one process driving n_gpus GPUs: -> /dev/null, then -> a tmpfs file."""
    exe = os.path.join(g2p.BIN_DIR, "gaf2paf")
    env = dict(os.environ, G2P_GPUS=str(n_gpus), G2P_STATS="1")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    res = {"gpus": n_gpus, "input": "tmpfs file, %d B" % in_bytes, "cmd": "G2P_GPUS=%d bin/gaf2paf -l lengths.tsv in.gaf" % n_gpus}

    def once(sink):
        t0 = time.perf_counter()
        with open(sink, "wb") as so:
            p = subprocess.run([exe, "-l", lengths_path, gaf_path], stdout=so, stderr=subprocess.PIPE, env=env)
        wall = time.perf_counter() - t0
        m = re.search(r"records=(\d+) in=(\d+) B out=(\d+) B device=([\d.]+) ms wall=([\d.]+) s", p.stderr.decode("latin-1"))
        if p.returncode != 0 or not m:
            raise RuntimeError("gaf2paf rc %d: %s" % (p.returncode, p.stderr.decode("latin-1")[-300:]))
        return wall, float(m.group(5)), int(m.group(1)), int(m.group(3))

    once("/dev/null")   # warm the page cache of the executable / library
    runs = [once("/dev/null") for _ in range(3)]
    wall, inner, nrec, nout = min(runs, key=lambda r: r[1])
    assert nrec == n_records, (nrec, n_records)
    res.update({"to_devnull": {"wall_s_process": wall, "wall_s_after_context_creation": inner, "records_per_s": nrec / inner,
                               "input_GBps": in_bytes / inner / 1e9, "out_bytes": nout}})
    try:
        st = os.statvfs(out_dir)
        if st.f_bavail * st.f_frsize > nout * 1.1 + (256 << 20):
            sink = os.path.join(out_dir, "g2p_bench_out_%d.paf" % os.getpid())
            try:
                runs = [once(sink) for _ in range(2)]
                wall, inner, nrec, nout = min(runs, key=lambda r: r[1])
                res["to_tmpfs_file"] = {"wall_s_process": wall, "wall_s_after_context_creation": inner, "records_per_s": nrec / inner}
            finally:
                if os.path.exists(sink):
                    os.unlink(sink)
    except Exception as ex:
        res["to_tmpfs_file"] = {"error": str(ex)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="short", choices=sorted(WORKLOADS))
    ap.add_argument("--records", type=int, default=0, help="records per GPU (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    if a.impl == "reference":
        return run_reference(a)

    import torch
    import torch.distributed as dist
    import cactus_gfa_tools_b200 as g2p
    import helpers as H

    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; this path has no CPU fallback (use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on STDOUT when the first communicator is created (measured on the
        # GPU box with NCCL_DEBUG=VERSION in the environment).  stdout carries the JSON line only: file
        # descriptor 1 points at stderr while the process group and its first collective come up.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_int(v):
        if world == 1:
            return [int(v)]
        t = torch.zeros(world, dtype=torch.int64, device="cuda")
        t[rank] = int(v)
        dist.all_reduce(t)
        return [int(x) for x in t.tolist()]

    def max_float(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl = WORKLOADS[a.workload]
    nrec = a.records or wl["records"]
    unstable = wl.get("kind") == "unstable"
    cv = g2p.Converter(local)
    threads = max(1, (os.cpu_count() or 8) // max(1, world))
    if unstable:
        # stable-interval GAF + rGFA (tests/helpers.py gen_rgfa_case, minigraph-like, node-aligned intervals); every rank
        # holds one copy of the same block, the logical input is the block repeated `world` times
        rgfa, block = H.gen_rgfa_case(7, n_contigs=24, n_records=nrec, aligned=True)
        t0 = time.perf_counter()
        ok, code, msg = cv.load_rgfa(rgfa)
        assert ok, msg
        table_load_s = time.perf_counter() - t0
        lengths = cv.node_lengths()
        keep_block = ctypes.create_string_buffer(block, len(block))
        addr, gen_bytes = ctypes.addressof(keep_block), len(block)
        a.no_cli = True   # the reference's interface for this path is two executables and a pipe
        dev_call, host_call = cv.unstable_convert_device, cv.unstable_convert_host_raw
    else:
        p = H.preset(wl["preset"], seed=1)
        lengths = H.gen_lengths(p)
        t0 = time.perf_counter()
        assert cv.load_lengths(lengths)
        table_load_s = time.perf_counter() - t0
        # ---- ONE logical input: rank r generates records [r*nrec, (r+1)*nrec) into a shared tmpfs file at its byte
        # offset; the file is then cut into `world` newline-aligned byte ranges and rank r takes range r.
        addr, gen_bytes = H.gen_records_raw(p, rank * nrec, nrec, threads=min(64, threads))
        dev_call, host_call = cv.convert_device, cv.convert_host_raw
    sizes = gather_int(gen_bytes)
    total_in = sum(sizes)
    want_cli = not a.no_cli
    shared = None
    port = os.environ.get("MASTER_PORT", "0")
    if world > 1 or want_cli:
        d = scratch_dir(total_in)
        shared = os.path.join(d, "g2p_bench_%s_%s_%d.gaf" % (port, a.workload, world))
        if rank == 0:
            with open(shared, "wb") as f:
                f.truncate(total_in)
        barrier()
        with open(shared, "r+b") as f:
            mm = mmap.mmap(f.fileno(), total_in)
            c0 = ctypes.c_char.from_buffer(mm)
            base = ctypes.addressof(c0)
            del c0   # (an exported buffer would keep the map from closing; the address stays valid while it is mapped)
            ctypes.memmove(base + sum(sizes[:rank]), addr, gen_bytes)
            mm.flush()
            barrier()
            a_off, b_off = g2p.shard_ranges(mm, world)[rank]
            nbytes = b_off - a_off
            pinned = g2p.lib.g2p_host_alloc(nbytes + 16)
            ctypes.memmove(pinned, base + a_off, nbytes)
            mm.close()
    else:
        a_off, nbytes = 0, gen_bytes
        pinned = g2p.lib.g2p_host_alloc(nbytes + 16)
        ctypes.memmove(pinned, addr, nbytes)
    if not unstable:
        H.gen_free(addr)
    d_in = torch.empty(nbytes + 16, dtype=torch.uint8, device="cuda")
    assert g2p.lib.g2p_copy_to_device(d_in.data_ptr(), pinned, nbytes) == 0
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream

    # ---- device-resident timing (value)
    res = None
    for _ in range(a.warmup):
        d_out, res = dev_call(d_in.data_ptr(), nbytes, stream)
    assert g2p.exit_code(res) == 0, "synthetic workload must convert cleanly"
    out_bytes = res.out_bytes
    n_records = res.n_records
    rec_all = gather_int(n_records)
    out_all = gather_int(out_bytes)
    in_all = gather_int(nbytes)
    assert sum(in_all) == total_in, "the shards must cover the logical input exactly"
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = {k: [] for k in ("emit_ms", "size_ms", "index_ms", "device_ms", "fused_ms", "unstable_ms", "par_ms")}
    launches = 0
    e0.record()
    for _ in range(a.steps):
        d_out, res = dev_call(d_in.data_ptr(), nbytes, stream)
        for k in ms:
            ms[k].append(getattr(res, k, 0.0))
        launches += res.gpu_launches
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    t_ms = max_float(e0.elapsed_time(e1))
    if a.dump_outputs:
        # before the e2e calls below, which reuse the converter's output buffer
        dump_outputs(a.dump_outputs, g2p, d_out, res, "_rank%d" % rank if world > 1 else "")

    # ---- end to end through the host-buffer C-ABI call (pinned input, H2D + D2H inside); the per-rank results
    # stay in per-rank pinned buffers whose rank order is the record order (a gather list, what writev consumes)
    e2e = None
    if not a.no_e2e:
        for _ in range(2):
            host_call(pinned, nbytes)
        barrier()
        w0 = time.perf_counter()
        for _ in range(a.steps):
            o_addr, r2 = host_call(pinned, nbytes)
        torch.cuda.synchronize()
        w_s = max_float(time.perf_counter() - w0)
        assert r2.out_bytes == out_bytes
        e2e = {"value": sum(rec_all) * a.steps / w_s, "unit": "records/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(r2.out_bytes),
               "ms_per_step": 1000.0 * w_s / a.steps, "input_GBps": total_in * a.steps / w_s / 1e9,
               "cold": {"table_load_s": table_load_s, "note": "g2p_load_lengths (host table build + upload) runs once per context, before the timed region"}}
    barrier()

    # ---- the drop-in executable on the same logical input (rank 0; the other ranks wait at the barrier)
    cli = None
    if want_cli and rank == 0:
        try:
            lp = shared + ".lengths.tsv"
            open(lp, "wb").write(lengths)
            try:
                cli = run_cli(g2p, shared, lp, world, sum(rec_all), total_in, os.path.dirname(shared))
            finally:
                os.unlink(lp)
        except Exception as ex:
            cli = {"error": str(ex)[-400:]}
    barrier()
    if shared and rank == 0 and os.path.exists(shared):
        os.unlink(shared)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = peaks()
    tot_rec, tot_out = sum(rec_all), sum(out_all)
    value = tot_rec * a.steps / (t_ms / 1000.0)
    mean = {k: statistics.mean(v) for k, v in ms.items()}
    n_fused = int(getattr(res, "n_fused", 0))
    short_kernel = "k_short<8>" if os.environ.get("G2P_SIZE_KERNEL") == "short" else "k_rec"
    # dominant kernel and its algorithmic bytes (DESIGN.md §4): the fused kernel reads the GAF and writes the PAF;
    # the two-pass pipeline's emit kernel does the same from descriptors, its size pass reads the GAF
    if mean["fused_ms"] > 0 and mean["fused_ms"] >= max(mean["size_ms"], mean["emit_ms"]):
        dom, dom_ms, dom_bytes, dom_key = "k_fuse (index + parse + look-back + format + store, one pass)", mean["fused_ms"], nbytes + out_bytes, "k_fuse"
    elif mean["emit_ms"] >= mean["size_ms"]:
        dom, dom_ms, dom_bytes, dom_key = "k_emit_lines (emit pass)", mean["emit_ms"], nbytes + out_bytes, "k_emit_lines"
    else:
        kname = ("k_par" if res.n_par * 2 > res.n_long else "k_long") if res.n_long * 2 > n_records else short_kernel
        dom, dom_ms, dom_bytes, dom_key = kname + " (size pass)", mean["size_ms"], nbytes, kname.split("<")[0] + "_size"
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        per_rec = tj.get(a.workload, {}).get(dom_key)
        if per_rec:
            traffic = per_rec * n_records
    except Exception:
        pass
    achieved = dom_bytes / (dom_ms / 1000.0) / 1e9 if dom_ms > 0 else 0.0
    line = {
        "metric": "gaf2paf_records_per_s", "value": value, "unit": "records/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": t_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic",
        "config": {"workload": wl["desc"], "preset": wl["preset"], "records": tot_rec, "gaf_bytes": total_in, "paf_bytes": tot_out,
                   "records_per_gpu": rec_all, "gaf_bytes_per_gpu": in_all, "table_entries": int(cv.table_entries), "l2": "inputs_larger_than_l2",
                   "sharding": "one logical input (shared tmpfs file), %d newline-aligned byte range(s), one per GPU, outputs in rank order = record order, no collective on the data path" % world},
        "input_GBps": total_in * a.steps / (t_ms / 1000.0) / 1e9,
        "pipeline_in_plus_out_GBps": (total_in + tot_out) * a.steps / (t_ms / 1000.0) / 1e9,
        "pipeline_frac_of_hbm_peak": (nbytes + out_bytes) * a.steps / (t_ms / 1000.0) / 1e9 / peak,
        "kernel_ms": {"index": mean["index_ms"], "size": mean["size_ms"], "emit": mean["emit_ms"], "fused": mean["fused_ms"], "par": mean["par_ms"],
                      "gaf2unstable_stage": mean["unstable_ms"], "device_pipeline": mean["device_ms"]},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "algorithmic_bytes_per_launch": dom_bytes, "peak_source": peak_src},
        "records_by_kernel": {"k_fuse": n_fused, short_kernel.split("<")[0]: int(n_records - res.n_long - n_fused) if n_fused == 0 else 0,
                              "k_par": int(res.n_par), "k_long": int(res.n_long - res.n_par - res.n_delegated), "general": int(res.n_delegated)},
        "gpu_launches": launches,
        "clocks": clocks,
        "table_load_s": table_load_s,
    }
    if e2e:
        line["e2e"] = e2e
    if cli:
        line["cli"] = cli
    if not a.no_cpu_baseline and world == 1:
        try:
            arm = CpuArm(H, wl["preset"], 1 if wl["preset"] else 7, wl["cpu_records"] * (2 if a.workload == "short" else 1), 1)
            try:
                line["cpu_baseline"] = arm.result([arm.step()])
            finally:
                arm.close()
        except Exception as ex:   # the baseline must not take the GPU number down with it
            line["cpu_baseline"] = {"error": str(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
