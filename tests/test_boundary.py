"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol
include/g2p.h declares, fails loudly without a GPU, and the host-side sharding logic
(newline-aligned byte ranges, ordered concatenation) is right — including a
world_size-2 gloo run of the multi-GPU partitioning."""
import os
import re
import subprocess
import sys

import pytest

import helpers as H

ROOT = H.ROOT


def test_header_symbols_exported(g2p):
    hdr = open(os.path.join(ROOT, "include", "g2p.h")).read()
    declared = set(re.findall(r"\b(g2p_[a-z_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    assert declared == set(g2p.EXPORTED_SYMBOLS)
    for s in declared:
        assert hasattr(g2p.lib, s), s


def test_no_cpu_fallback_without_gpu(g2p):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(g2p.G2PError):
        g2p.Converter(0)


def test_cli_without_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    exe = os.path.join(ROOT, "cactus-gfa-tools_b200", "bin", "gaf2paf")
    d = H.golden("gaf2paf_kat.json")
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        open(lp, "w").write(d["lengths"])
        rc, out, err = H.run_tool(exe, ["-", "-l", lp], b"")
        assert rc == 1 and out == b"" and "no usable CUDA device" in err


def test_cli_usage_errors_match_reference():
    """Argument handling happens before any GPU use, so it is checkable on CPU."""
    exe = os.path.join(ROOT, "cactus-gfa-tools_b200", "bin", "gaf2paf")
    cases = [[], ["x.gaf"], ["-l", "/nonexistent/l.tsv", "x.gaf"], ["-h"], ["-l"], ["--lengths"], ["-z", "a"]]
    for args in cases:
        rc, out, err = H.run_tool(exe, args)
        assert rc == 1 and out == b"", args
        rrc, rout, rerr = H.reference_cli("gaf2paf", args, {})
        assert rrc == rc, args
        assert rerr == err.replace(exe, "X"), args


def test_shard_ranges(g2p):
    p = H.preset("short", seed=3)
    gaf = H.gen_records(p, 0, 500, threads=2)
    for n in (1, 2, 3, 8, 64):
        rs = g2p.shard_ranges(gaf, n)
        assert len(rs) == n and rs[0][0] == 0 and rs[-1][1] == len(gaf)
        for (a, b), (c, d) in zip(rs, rs[1:]):
            assert b == c
        for a, b in rs:
            assert a == b or gaf[b - 1:b] == b"\n" or b == len(gaf)
            assert a == 0 or gaf[a - 1:a] == b"\n"
    # fewer lines than shards
    rs = g2p.shard_ranges(b"abc\n", 4)
    assert b"".join(b"abc\n"[a:b] for a, b in rs) == b"abc\n"


_GLOO = r"""
import os, sys, hashlib
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import torch, torch.distributed as dist
import helpers as H
import cactus_gfa_tools_b200 as g2p
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
p = H.preset("short", seed=5)
gaf = H.gen_records(p, 0, 400, threads=1)
lengths = H.gen_lengths(p)
a, b = g2p.shard_ranges(gaf, world)[rank]
rc, out, err, kind = H.run_gaf2paf_cpu(gaf[a:b], lengths, kind="port")   # CPU stand-in for the per-rank GPU call
assert rc == 0
# ordered concatenation on rank 0 (what the host driver does with per-GPU outputs)
sizes = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
dist.all_gather(sizes, torch.tensor([len(out)], dtype=torch.int64))
mx = int(max(s.item() for s in sizes))
pad = torch.zeros(mx, dtype=torch.uint8); pad[:len(out)] = torch.frombuffer(bytearray(out), dtype=torch.uint8)
parts = [torch.zeros(mx, dtype=torch.uint8) for _ in range(world)]
dist.all_gather(parts, pad)
if rank == 0:
    whole = b"".join(bytes(parts[i][:int(sizes[i].item())].numpy()) for i in range(world))
    rc2, ref, _, _ = H.run_gaf2paf_cpu(gaf, lengths, kind="port")
    assert whole == ref, "sharded output differs from unsharded"
    print("GLOO_OK", hashlib.md5(whole).hexdigest())
dist.barrier()
"""


def test_two_rank_sharding_gloo(tmp_path):
    script = tmp_path / "gloo_shard.py"
    script.write_text(_GLOO % {"root": ROOT})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29531", str(script)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, timeout=300)
    assert p.returncode == 0 and b"GLOO_OK" in p.stdout, p.stdout.decode()[-2000:]
