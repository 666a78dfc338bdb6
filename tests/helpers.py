"""Shared test / bench helpers: synthetic generator binding, oracle runners, golden vectors.

Everything here is test infrastructure.  The oracle (oracle/bin/*, oracle/_ref/*) is only
ever used as the checker or as the timed CPU baseline — never by the product path."""
import ctypes
import json
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE_BIN = os.path.join(ROOT, "oracle", "bin")
REF_BIN = os.path.join(ROOT, "oracle", "_ref")
BUILD = os.path.join(ROOT, "build")


class GenParams(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64)] + [(k, ctypes.c_uint32) for k in (
        "n_nodes", "node_len_lo", "node_len_hi", "steps_lo", "steps_hi", "mrun_lo", "mrun_hi", "indel_lo", "indel_hi",
        "max_runs", "pct_rev", "pct_minus", "use_eqx", "stable", "qlen_min", "pct_star", "mix_every", "qname_len", "extra_tag_len")]


_gen = None


def gen_lib():
    global _gen
    if _gen is None:
        path = os.path.join(BUILD, "libgafgen.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", ROOT, "build/libgafgen.so"], stdout=subprocess.DEVNULL)
        _gen = ctypes.CDLL(path)
        _gen.gafgen_preset.argtypes = [ctypes.c_char_p, ctypes.POINTER(GenParams)]
        _gen.gafgen_preset.restype = None
        _gen.gafgen_lengths.argtypes = [ctypes.POINTER(GenParams), ctypes.c_void_p, ctypes.c_size_t]
        _gen.gafgen_lengths.restype = ctypes.c_size_t
        _gen.gafgen_records.argtypes = [ctypes.POINTER(GenParams), ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
        _gen.gafgen_records.restype = ctypes.c_size_t
        _gen.gafgen_records_alloc.argtypes = [ctypes.POINTER(GenParams), ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.POINTER(ctypes.c_size_t)]
        _gen.gafgen_records_alloc.restype = ctypes.c_void_p
        _gen.gafgen_free.argtypes = [ctypes.c_void_p]
        _gen.gafgen_free.restype = None
    return _gen


def preset(name, seed=1, **over):
    p = GenParams()
    gen_lib().gafgen_preset(name.encode(), ctypes.byref(p))
    if p.n_nodes == 0:
        raise ValueError("unknown preset " + name)
    p.seed = seed
    for k, v in over.items():
        setattr(p, k, v)
    return p


def gen_lengths(p):
    n = gen_lib().gafgen_lengths(ctypes.byref(p), None, 0)
    buf = ctypes.create_string_buffer(n)
    gen_lib().gafgen_lengths(ctypes.byref(p), buf, n)
    return buf.raw


def gen_records_raw(p, first, count, threads=None):
    """-> (address, size) of a malloc'd buffer; release with gen_free(address)."""
    threads = threads or min(32, os.cpu_count() or 1)
    n = ctypes.c_size_t()
    addr = gen_lib().gafgen_records_alloc(ctypes.byref(p), first, count, threads, ctypes.byref(n))
    if not addr:
        raise MemoryError("gafgen_records_alloc")
    return addr, n.value


def gen_free(addr):
    gen_lib().gafgen_free(addr)


def gen_records(p, first, count, threads=None):
    addr, n = gen_records_raw(p, first, count, threads)
    try:
        return ctypes.string_at(addr, n)
    finally:
        gen_free(addr)


def gen_records_into(p, first, count, addr, cap, threads=None):
    """Generate straight into a caller buffer (e.g. pinned memory); returns the byte count
    (nothing written if it exceeds cap)."""
    threads = threads or min(32, os.cpu_count() or 1)
    return gen_lib().gafgen_records(ctypes.byref(p), first, count, addr, cap, threads)


def oracle_path(kind="auto", tool="gaf2paf"):
    """Path of the checker binary of `tool` (gaf2paf, gaf2unstable, gaffilter): the unmodified reference build when
    present (kind 'reference'), else the restatement oracle/bin/<tool>_oracle (kind 'port')."""
    ref = os.path.join(REF_BIN, tool)
    port = os.path.join(ORACLE_BIN, tool + "_oracle")
    if kind in ("auto", "reference") and os.path.exists(ref):
        return ref, "reference"
    if kind == "reference":
        raise FileNotFoundError(ref)
    if not os.path.exists(port):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    return port, "port"


def run_tool(binary, args, stdin_bytes=None):
    p = subprocess.run([binary] + list(args), input=stdin_bytes, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    rc = p.returncode
    if rc < 0:
        rc = 128 - rc
    return rc, p.stdout, p.stderr.decode("latin-1")


def run_gaf2paf_cpu(gaf, lengths, kind="auto"):
    """Run the CPU checker on in-memory inputs -> (rc, stdout bytes, stderr text, kind)."""
    binary, k = oracle_path(kind)
    with tempfile.TemporaryDirectory() as td:
        lp = os.path.join(td, "l.tsv")
        with open(lp, "wb") as f:
            f.write(lengths)
        rc, out, err = run_tool(binary, ["-", "-l", lp], gaf)
    return rc, out, err, k


def golden(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def reference_cli(tool, args, subst):
    """(exit code, stdout, stderr) of the reference `tool` on a command line it rejects, its own path written X in stderr:
    the reference build when present, else the run stored in tests/golden/reference_runs.json.  `args` may hold the
    placeholders of that file ({L}, {A}, {G}); `subst` maps them to paths."""
    ref = os.path.join(REF_BIN, tool)
    if os.path.exists(ref):
        rc, out, err = run_tool(ref, [subst.get(a, a) for a in args])
        return rc, out, err.replace(ref, "X")
    for r in golden("reference_runs.json")["cli"][tool]:
        if r["args"] == list(args):
            err = r["err"]
            for k, v in subst.items():
                err = err.replace(k, v)
            return r["rc"], r["out"].encode("latin-1"), err
    raise KeyError("no stored %s run for %r: add it to tests/golden/make_reference_runs.py" % (tool, args))


# ---- gaf2unstable: synthetic rGFA + stable-coordinate GAF (BASELINE config 2 shape) -------------
def gen_rgfa_case(seed, n_contigs=4, n_records=500, aligned=False, multi_ref_pct=3):
    """Returns (rgfa bytes, gaf bytes).  Rank-0 chains over `n_contigs` reference contigs (one with an
    "id=..|" SN prefix), rank-1 bubble nodes on non-reference contigs, and minigraph-like GAF records
    whose path steps are stable intervals (`aligned`: intervals coincide with node boundaries, as
    minigraph emits them, so that the output is valid input for gaf2paf), whole-contig paths,
    unmapped records and '*' lines."""
    import random
    rnd = random.Random(seed)
    lines, contigs = [], []          # contigs: (sn, [(name, off, len)])
    nid = 1
    links = []
    for c in range(n_contigs):
        sn = ("id=HG%d|chr%d" % (c, c + 1)) if c == 1 else "chr%d" % (c + 1)
        nodes, off = [], 0
        for _ in range(rnd.randrange(8, 40)):
            ln = rnd.randrange(20, 300)
            nodes.append(("s%d" % nid, off, ln)); nid += 1
            off += ln
        contigs.append((sn, nodes))
    bubbles = []
    for c, (sn, nodes) in enumerate(contigs):
        for k in range(rnd.randrange(1, 4)):
            i = rnd.randrange(0, len(nodes) - 2)
            ln = rnd.randrange(20, 200)
            bsn = "HG00%d#1#ctg%d_%d" % (c, c, k)
            boff = rnd.randrange(0, 5000)
            bubbles.append((bsn, [("s%d" % nid, boff, ln)], nodes[i][0], nodes[i + 2][0]))
            nid += 1
    def seq(n):
        return "".join(rnd.choice("ACGT") for _ in range(n))
    for sn, nodes in contigs:
        for j, (name, off, ln) in enumerate(nodes):
            lines.append("S\t%s\t%s\tLN:i:%d\tSN:Z:%s\tSO:i:%d\tSR:i:0" % (name, seq(ln), ln, sn, off))
            if j:
                links.append("L\t%s\t+\t%s\t+\t0M\tSR:i:0\tL1:i:%d\tL2:i:%d" % (nodes[j - 1][0], name, nodes[j - 1][2], ln))
    for bsn, bn, left, right in bubbles:
        name, off, ln = bn[0]
        lines.append("S\t%s\t%s\tLN:i:%d\tSN:Z:%s\tSO:i:%d\tSR:i:1" % (name, seq(ln), ln, bsn, off))
        links.append("L\t%s\t+\t%s\t+\t0M\tSR:i:1\tL1:i:1\tL2:i:%d" % (left, name, ln))
        links.append("L\t%s\t+\t%s\t+\t0M\tSR:i:1\tL1:i:%d\tL2:i:1" % (name, right, ln))
    rgfa = ("\n".join(lines + links) + "\n").encode()
    allc = contigs + [(b[0], b[1]) for b in bubbles]

    def interval(sn, nodes):
        lo, hi = nodes[0][1], nodes[-1][1] + nodes[-1][2]
        if aligned:
            i = rnd.randrange(len(nodes))   # minigraph's stable steps are exactly one node each
            return nodes[i][1], nodes[i][1] + nodes[i][2]
        s = rnd.randrange(lo, hi - 1)
        return s, rnd.randrange(s + 1, min(hi, s + 900) + 1)

    recs = []
    for r in range(n_records):
        x = rnd.random()
        tags = rnd.sample(["tp:A:P", "cm:i:%d" % rnd.randrange(100), "s1:i:%d" % rnd.randrange(500), "dv:f:0.0123", "rc:Z:old", "zd:i:3"],
                          rnd.randrange(0, 5))
        mapq = rnd.choice([0, 1, 60, 255, 300])
        strand = rnd.choice("+-")
        if x < 0.02:
            recs.append("*\t>s43\t97\t12\t0\t6\t92")
            continue
        if x < 0.05 and not aligned:   # unmapped record: no cg tag, gaf2paf would stop on it
            recs.append("\t".join(["q%d" % r, "200", "0", "60", "+", "*", "*", "*", "*", "*", "*", "255"] + tags))
            continue
        if x < 0.20:   # whole-contig path
            sn, nodes = rnd.choice(contigs)
            s, e = interval(sn, nodes)
            plen = nodes[-1][1] + nodes[-1][2]
            W = e - s
            cg = "cg:Z:%dM" % W
            cols = ["q%d" % r, str(W + 20), "5", str(5 + W), strand, sn, str(plen), str(s), str(e), str(W), str(W), str(mapq)]
        else:
            ci = rnd.randrange(len(contigs))
            steps, total, lens = [], 0, []
            for k in range(rnd.randrange(1, 7)):
                pool = contigs[ci:ci + 1] + [(b[0], b[1]) for b in bubbles if b[0].startswith("HG00%d#" % ci)]
                if rnd.random() * 100 < multi_ref_pct:
                    pool = allc
                sn, nodes = rnd.choice(pool)
                s, e = interval(sn, nodes)
                steps.append("%s%s:%d-%d" % (rnd.choice("><"), sn, s, e))
                lens.append(e - s); total += e - s
            ps = rnd.randrange(0, lens[0])
            pe = total - rnd.randrange(0, lens[-1]) if len(lens) > 1 else rnd.randrange(ps + 1, total + 1)
            if pe <= ps:
                ps, pe = 0, total
            W = pe - ps
            a = rnd.randrange(1, W) if W > 3 else W
            cg = "cg:Z:%dM" % W if a == W else "cg:Z:%dM2I%dM" % (a, W - a)
            q = W + (0 if a == W else 2)
            cols = ["q%d" % r, str(q + 20), "5", str(5 + q), strand, "".join(steps), str(total), str(ps), str(pe), str(W), str(q), str(mapq)]
        pos = rnd.randrange(0, len(tags) + 1)
        recs.append("\t".join(cols + tags[:pos] + [cg] + tags[pos:]))
    return rgfa, ("\n".join(recs) + "\n").encode()


def run_gaf2unstable_ref(gaf, rgfa, want_lengths=False):
    """The reference gaf2unstable (oracle/_ref) on in-memory inputs -> (rc, stdout, stderr[, node-lengths])."""
    binary, _kind = oracle_path("auto", "gaf2unstable")   # reference build when present, else the restatement
    with tempfile.TemporaryDirectory() as td:
        gp, lp = os.path.join(td, "g.gfa"), os.path.join(td, "nl.tsv")
        with open(gp, "wb") as f:
            f.write(rgfa)
        rc, out, err = run_tool(binary, ["-", "-g", gp] + (["-o", lp] if want_lengths else []), gaf)
        if want_lengths:
            return rc, out, err, open(lp, "rb").read() if os.path.exists(lp) else b""
    return rc, out, err


# ---- gaffilter: records whose query intervals overlap (several alignments per query, primary / secondary, mixed mapq) ----
def gen_filter_case(seed, n_records=3000, n_queries=150, paf=False):
    """GAF (or, paf=True, the PAF that gaf2paf makes of it: -> (text, lengths)) in which many records share a query name,
    so that gaffilter has overlaps to resolve."""
    import random
    rnd = random.Random(seed)
    p = preset("short", seed=seed)
    lengths = gen_lengths(p)
    lines = gen_records(p, 0, n_records, threads=1).split(b"\n")[:-1]
    out = []
    for i, ln in enumerate(lines):
        f = ln.split(b"\t")
        f[0] = b"q%d" % rnd.randrange(n_queries)
        if rnd.random() < 0.3:
            f = [x if not x.startswith(b"tp:A:") else b"tp:A:S" for x in f]
        if rnd.random() < 0.1:
            f = [x for x in f if not x.startswith(b"tp:A:")]
        f[11] = str(rnd.choice([0, 1, 5, 20, 60, 255])).encode()
        if rnd.random() < 0.2:
            f.insert(12, b"rc:Z:chr%d" % rnd.randrange(3))
        out.append(b"\t".join(f))
        if rnd.random() < 0.01:
            out.append(b"*\t>s43\t97\t12\t0\t6\t92")
    gaf = b"\n".join(out) + b"\n"
    if not paf:
        return gaf, lengths
    rc, paf_text, err, kind = run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0, err
    return paf_text, lengths


def gen_spread_filter_case(seed, n_records=6000, n_queries=3, depth=4, paf=False):
    """Like gen_filter_case, but with few query sequences whose records lie along the whole query (assembly contigs mapped
    in pieces): each record's query interval moves by a random offset, about `depth` records cover a query position."""
    import random
    rnd = random.Random(seed)
    gaf, lengths = gen_filter_case(seed, n_records=n_records, n_queries=n_queries)
    span = max(1, n_records // n_queries * 120 // depth)
    out = []
    for ln in gaf.split(b"\n")[:-1]:
        f = ln.split(b"\t")
        if f[0] != b"*":
            off = rnd.randrange(span)
            f[1] = b"%d" % (int(f[1]) + span)
            f[2] = b"%d" % (int(f[2]) + off)
            f[3] = b"%d" % (int(f[3]) + off)
        out.append(b"\t".join(f))
    gaf = b"\n".join(out) + b"\n"
    if not paf:
        return gaf
    rc, paf_text, err, kind = run_gaf2paf_cpu(gaf, lengths)
    assert rc == 0, err
    return paf_text
