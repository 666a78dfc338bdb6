"""The PAF line writer of k_emit_lines and k_long at the shapes of its pieces, under the SIMT emulator.

k_emit_lines<false> (k_rec's lines) prints the verbatim middle of the cut CIGAR with one flat loop that finds the token
ends from a rolling mask of the op letters (put_tokens); k_emit_lines<true> (k_par's lines) and k_long keep the byte
loops.  These cases put the pieces at the lengths where that code changes step: CIGAR middles of one token and of many
(longer than several 4-byte words and than the 12-byte letter window), op lengths of 1 to 7 digits, every direction
(+/- record x >/< step), query names of 3 to 36 bytes, tp / rc values of 2 to 12 bytes or absent, MAPQ '*' and 255,
and warps whose 32 lines are longer than k_emit_lines<false>' staging buffer.  The bytes must equal the reference's,
and the records must have been converted by the kernels the configuration names."""
import os
import random
import tempfile

import pytest

import helpers as H
from test_convert_limits import SIMT, SIMT_LONG, run_simt, oracle

PAD = "zz:Z:" + "y" * 240   # pushes a record past k_rec's 240 bytes: k_par (or k_long with G2P_PAR=0) takes it

CONFIGS = {   # name -> (binary, environment, pad)
    "rec": (SIMT, {"G2P_FUSE": "0"}, False),
    "par": (SIMT, {"G2P_FUSE": "0"}, True),
    "long": (SIMT, {"G2P_FUSE": "0", "G2P_PAR": "0"}, True),
    "slong": (SIMT_LONG, {"G2P_FUSE": "0", "G2P_PAR": "0"}, False),
}


def cigar(rng, target, ntok, maxd):
    """A CIGAR of about ntok tokens that consumes exactly `target` reference bases; op lengths of up to maxd digits."""
    cuts = sorted(rng.sample(range(1, target), min(ntok - 1, target - 1))) if ntok > 1 else []
    parts = [b - a for a, b in zip([0] + cuts, cuts + [target])]
    out = []
    for i, x in enumerate(parts):
        if i and rng.random() < 0.3:
            out.append("%d%s" % (rng.randint(1, 10 ** rng.randint(1, maxd) - 1), "I"))
        out.append("%d%s" % (x, rng.choice("MMM=XD") if 0 < i < len(parts) - 1 else "M"))
    return "".join(out)


def make_case(seed, big=False):
    rng = random.Random(seed)
    nodes = {"n%d" % i: rng.randint(2_000_000, 20_000_000) if big else rng.randint(30, 400) for i in range(12)}
    lengths = "".join("%s\t%d\n" % kv for kv in nodes.items())
    recs = []
    for r in range(rng.randint(40, 120)):
        ns = rng.randint(1, 4)
        steps = [(rng.choice("<>"), rng.choice(list(nodes))) for _ in range(ns)]
        total = sum(nodes[n] for _, n in steps)
        ps = rng.randint(0, nodes[steps[0][1]] // 2)
        pe = total - rng.randint(0, nodes[steps[-1][1]] // 2)
        ntok = rng.choice([1, 2, 3, 5, 9, 16, 24, 30])
        cg = cigar(rng, pe - ps, ntok, 7 if big else 3)
        q = sum(int(t[:-1]) for t in __import__("re").findall(r"\d+[MI=X]", cg))
        qs = rng.randint(0, 50)
        mapq = rng.choice(["*", "255", "0", "60", "254"])
        tags = [rng.choice(["", "tp:A:P", "tp:Z:", "tp:Z:ab", "tp:Z:abcdefghij"]),
                rng.choice(["", "rc:Z:x", "rc:i:1234", "rc:Z:0123456789"])]
        qn = "q%d_" % r + "x" * rng.choice([0, 1, 2, 3, 5, 12, 30])
        cols = [qn, qs + q + rng.randint(0, 9), qs, qs + q, rng.choice("+-"), "".join(o + n for o, n in steps), total,
                ps, pe, rng.randint(1, 9), rng.randint(10, 99), mapq]
        recs.append("\t".join(str(c) for c in cols + [t for t in tags if t] + ["cg:Z:" + cg]))
    return lengths, recs


def routed(cfg, st, n):
    _, nrec, to_par, steps, to_long, general = st
    if cfg == "rec":   # k_rec takes most of them (records much longer than the mean go on to k_par)
        return to_par < n and general == 0
    if cfg == "par":
        return to_par == n and to_long < n and general == 0
    return to_long == (n if cfg == "long" else nrec) and general == 0


@pytest.mark.parametrize("cfg", list(CONFIGS))
@pytest.mark.parametrize("seed,big", [(1, False), (2, False), (3, True)])
def test_pieces_match_reference(cfg, seed, big):
    binary, env, pad = CONFIGS[cfg]
    lengths, recs = make_case(seed, big)
    if cfg == "rec":
        recs = [r for r in recs if len(r) <= 240]
    if pad:
        recs = [r.replace("\tcg:Z:", "\t" + PAD + "\tcg:Z:", 1) for r in recs]
    data = ("\n".join(recs) + "\n").encode()
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        with open(lp, "w") as f:
            f.write(lengths)
        rc, ref, err = oracle(lp, data)
        assert rc == 0 and ref.count(b"\n") > len(recs), err[-300:]
        grc, out, st = run_simt(binary, env, lp, data)
    assert grc == rc and out == ref, "%s: %d vs %d bytes" % (cfg, len(out), len(ref))
    assert st[0] == "pipe" and routed(cfg, st, len(recs)), (cfg, st)
