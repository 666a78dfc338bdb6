"""gaf2unstable at its edges: a named table of hand-built records and rGFAs, each checked against the reference
gaf2unstable (oracle/_ref, or the independent restatement oracle/bin/gaf2unstable_oracle when it is absent).

The per-record code (g2u_core.cuh) computes offsets in int64 and keeps node lengths in u32.  The cases put numbers at
and around 2^31, 2^32, 2^53 and 2^62, intervals at and +-1 around every node boundary of contigs whose nodes are
contiguous, apart, overlapping, on a duplicate SO, or start past 0, and the text around every parse and tag-collection
limit.  What is compared: the exit code, stdout, the multi-contig warning text on stderr and the -o file.  Where the
reference aborts, the reference build may lose what is still in its stdio buffer (stdout is compared as a prefix), and
a zero-length interval makes it crash (139) where the port and this library abort (134).

CPU: every case alone between ordinary records, and all cases that do not abort together in three seeded orders (so
that one warp holds short, long, empty and warning records), under
  - g2u_hostsim: the per-record code compiled for the host;
  - g2u_simt: k_unstable -- the kernel the library runs -- under the SIMT emulator, over a grid of 3 CTAs of 64 threads
    so that its grid-stride loop takes several turns, and with the CTAs in reverse order; k_unstable_staged; the staged
    kernel with tiny staging buffers (g2u_simt_small);
  - gaf2unstable_stub: the executable's host logic on 1 and 3 contexts, in small chunks.
GPU (-m gpu): Converter.unstable_host and bin/gaf2unstable, and the fused unstable_convert_host against
`gaf2unstable | gaf2paf -l <its -o file>` of the checkers; the fused call's 4 GiB limit on its intermediate GAF and its
warning text; one g2p_unstable_host call whose output passes 4 GiB."""
import concurrent.futures
import hashlib
import os
import random
import subprocess
import tempfile

import pytest

import helpers as H

HOSTSIM = os.path.join(H.BUILD, "g2u_hostsim")
SIMT = os.path.join(H.BUILD, "g2u_simt")
STUB = os.path.join(H.BUILD, "gaf2unstable_stub")
CHUNK = "200"   # G2P_CHUNK_BYTES of the stub runs: about one record per chunk

RUNNERS = {
    "hostsim": (HOSTSIM, {}),
    "simt-list": (SIMT, {}),
    "simt-list-reverse": (SIMT, {"G2P_SIMT_REVERSE": "1"}),
    "simt-staged": (SIMT, {"G2U_SIMT_STAGED": "1"}),
    "simt-small": (SIMT + "_small", {}),
    "stub-1gpu": (STUB, {"G2P_GPUS": "1", "G2P_CHUNK_BYTES": CHUNK}),
    "stub-3gpus": (STUB, {"G2P_GPUS": "3", "G2P_CHUNK_BYTES": CHUNK}),
}
POOL = concurrent.futures.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))


# ---- the rGFA -------------------------------------------------------------------------------------------------
BASES = {"0": 0, "b31": 2**31 - 5, "b32": 2**32 - 5, "b53": 2**53, "b62": 2**62}
LAYOUTS = {   # (offset from the base, length) in file order
    "contiguous": [(0, 10), (10, 5), (15, 20)],
    "gaps": [(0, 10), (20, 5), (30, 8)],
    "overlaps": [(0, 10), (5, 10), (12, 6)],
    "dupso": [(0, 10), (10, 5), (10, 7), (15, 4)],   # std::set keeps the first node of an SO and drops the later one
    "past0": [(7, 10), (17, 5), (27, 3)],
    "single": [(0, 12)],
    "onebp": [(0, 1), (1, 1), (2, 1), (3, 1)],
}
NAMES = {   # contig names around the exact (<= 16 bytes) and hashed keys of the lengths table
    "n15": "c" * 14 + "1", "n16": "c" * 15 + "1", "n17": "c" * 16 + "1", "n40": "c" * 39 + "1",
    "n16b": "c" * 15 + "2", "n17b": "c" * 16 + "2", "n40b": "c" * 39 + "2",
    "chr1": "chr1", "chr10": "chr10", "pfx": "id=HG7|chrP", "pfx2": "id=HG8|chrP",
}
ORD = "chrO"   # the ordinary records' contig


def layout_contig(lay, bk):
    return "L_%s_%s" % (lay, bk)


class Graph:
    """An rGFA of rank-0 contigs: S lines of `A`*length with LN / SN / SO / SR tags, node names s1, s2, ..."""

    def __init__(self):
        self.lines, self.contigs, self.nid = [], {}, 0

    def contig(self, sn, nodes):
        out = []
        for off, ln in nodes:
            self.nid += 1
            name = "s%d" % self.nid
            self.lines.append("S\t%s\t%s\tLN:i:%d\tSN:Z:%s\tSO:i:%d\tSR:i:0" % (name, "A" * ln, ln, sn, off))
            out.append((name, off, ln))
        self.contigs[sn] = out
        return out

    def text(self):
        return ("\n".join(self.lines) + "\n").encode()


def main_graph():
    g = Graph()
    g.contig(ORD, [(0, 30), (30, 40), (70, 25)])
    for bk, base in BASES.items():
        for lay, nodes in LAYOUTS.items():
            g.contig(layout_contig(lay, bk), [(base + o, ln) for o, ln in nodes])
    for sn in NAMES.values():
        g.contig(sn, [(0, 8), (8, 8)])
    g.contig("chrZ", [(100, 50), (150, 50)])
    return g


# ---- records --------------------------------------------------------------------------------------------------
def rec(path, plen, ps, pe, qname="q", qlen=None, qs="0", qe=None, strand="+", m=None, b=None, mapq="60", tags=()):
    """One GAF line; numbers may be given as text.  Default columns make a record gaf2paf converts: cg = (pe - ps)M."""
    w = None
    try:
        w = int(pe) - int(ps)
    except ValueError:
        pass
    d = str(w) if w is not None else "1"
    cols = [qname, str(qlen if qlen is not None else d), str(qs), str(qe if qe is not None else d), strand, path,
            str(plen), str(ps), str(pe), str(m if m is not None else d), str(b if b is not None else d), str(mapq)]
    tg = list(tags)
    if not any(t.startswith("cg:") for t in tg) and w is not None and w >= 0:
        tg.append("cg:Z:%dM" % w)
    return "\t".join(cols + tg)


def ordinary(i):
    """A record on chrO that every tool converts: a step, or the bare contig."""
    s, e = [(0, 30), (30, 70), (5, 90), (70, 95)][i % 4]
    if i % 5 == 4:
        return rec(ORD, 95, s, e, qname="o%d" % i, tags=["tp:A:P"])
    return rec(">%s:%d-%d" % (ORD, s, e), e - s, 0, e - s, qname="o%d" % i, tags=["tp:A:P", "NM:i:0"])


def geometry_points(nodes):
    ends = sorted({o for _n, o, _l in nodes} | {o + ln for _n, o, ln in nodes})
    pts = {p + d for p in ends for d in (-1, 0, 1)}
    return sorted(pts | {ends[0] - 3, ends[-1] + 3})


def geometry_cases(g):
    """Interval geometry: every start and end at and +-1 around every node boundary, and before the first node and
    past the last, as a '>' step (also '<' at the bases 0 and 2^62) and as a bare contig whose ps / pe are rewritten."""
    cases = {}
    for bk in BASES:
        for lay in LAYOUTS:
            sn = layout_contig(lay, bk)
            pts = geometry_points(g.contigs[sn])
            base = BASES[bk]
            for s in pts:
                for e in pts:
                    if e < s:
                        continue
                    tag = "geo/%s/%s/%d-%d" % (lay, bk, s - base, e - base)
                    for d in (">", "<") if bk in ("0", "b62") else (">",):
                        cases[tag + d] = rec("%s%s:%d-%d" % (d, sn, s, e), e - s, 0, e - s)
                    if s < e and (lay in ("contiguous", "gaps", "dupso") or bk == "0"):
                        cases[tag + "/bare"] = rec(sn, 999, s, e)
            nodes = g.contigs[sn]
            cases["geo/%s/%s/bare-star-ps" % (lay, bk)] = rec(sn, 999, "*", nodes[0][1] + 3, tags=["cg:Z:4M"])
            cases["geo/%s/%s/bare-star-pe" % (lay, bk)] = rec(sn, 999, nodes[0][1], "*", tags=["cg:Z:4M"])
    return cases


BIG = ["123456789012345678", "9223372036854775807", "9223372036854775808", "-9223372036854775808",
       "-9223372036854775809", "12345678901234567890", "99999999999999999999"]


def text_cases():
    """The text of an interval, of columns 2-4 and 7-11, and of MAPQ."""
    c = layout_contig("contiguous", "0")
    cases = {}
    ivals = [(" 3", "12"), ("+3", "12"), ("003", "012"), ("3", "12x"), ("3x", "12"), ("3", "-0"), ("-0", "12"), ("3", ""),
             ("", "12"), ("3", " 12"), ("3", "+12"), ("3", "12 "), ("0", "35"), ("3", "3"), ("3", "2"),
             ("3", "000000000000000012"), ("3", "0000000000000000012"), ("3", "00000000000000000012")] + \
            [("3", v) for v in BIG] + [(v, "12") for v in BIG]
    for i, (s, e) in enumerate(ivals):
        cases["text/interval/%d/%r-%r" % (i, s, e)] = rec(">%s:%s-%s" % (c, s, e), 9, 0, 9)
    cases["text/interval/no-dash"] = rec(">%s:3" % c, 9, 0, 9)
    cases["text/interval/two-colons"] = rec(">%s:3:4-12" % c, 9, 0, 9)
    big = layout_contig("contiguous", "b62")
    for name, v in [("m1", "-1"), ("star", "*"), ("zero", "0"), ("neg2", "-2"), ("sp", " 7"), ("plus", "+7"), ("lz", "007"), ("junk", "7x")] + \
            [("big%d" % i, v) for i, v in enumerate(BIG)]:
        for col in ("qlen", "qs", "qe", "m", "b"):
            cases["text/col-%s/%s" % (col, name)] = rec(">%s:3-12" % c, 9, 0, 9, **{col: v})
        cases["text/col-plen/%s" % name] = rec(">%s:3-12" % c, v, 0, 9)
        cases["text/col-ps/%s" % name] = rec(">%s:3-12" % c, 9, v, 9)
        cases["text/col-pe/%s" % name] = rec(">%s:3-12" % c, 9, 0, v)
        cases["text/bare-ps/%s" % name] = rec(c, 35, v, 12)
        cases["text/bare-pe/%s" % name] = rec(c, 35, 3, v)
        cases["text/bare-b62-ps/%s" % name] = rec(big, 35, v, 2**62 + 12)
    for v in ["0", "1", "60", "254", "255", "256", "1000", "2147483647", "2147483648", "-2147483648", "-2147483649",
              "-1", "*", "**", "", " 60", "+60", "060", "60x", "9223372036854775808"]:
        cases["text/mapq/%r" % v] = rec(">%s:3-12" % c, 9, 0, 9, mapq=v)
    for v in ["", "++", "-", "*", "x", "+-"]:
        cases["text/strand/%r" % v] = rec(">%s:3-12" % c, 9, 0, 9, strand=v)
    cases["text/qname-empty"] = rec(">%s:3-12" % c, 9, 0, 9, qname="")
    cases["text/eleven-columns"] = "\t".join(rec(">%s:3-12" % c, 9, 0, 9).split("\t")[:11])
    cases["text/empty-path"] = rec("", 9, 0, 9)
    cases["text/star-path"] = rec("*", "*", "*", "*", m="*", b="*", tags=["tp:A:U"])
    cases["text/star-path-rc"] = rec("*", 5, 1, 2, tags=["rc:Z:keep", "aa:i:1"])
    cases["text/star-line"] = "*\t>s43\t97\t12\t0\t6\t92"
    cases["text/empty-line"] = ""
    cases["text/blank-tail"] = rec(">%s:3-12" % c, 9, 0, 9) + "\t"
    return cases


def tag_cases():
    """Optional fields: names that sort around rc, an input rc (replaced; kept when the path is '*' or spans several
    contigs), 16 and 17 fields around the collection limit, a field over 65 535 bytes, a name over 255 bytes, and
    duplicates on both sides of each limit."""
    c = layout_contig("contiguous", "0")
    step = ">%s:3-12" % c
    multi = ">%s:3-12>%s:%d-%d" % (c, layout_contig("contiguous", "b31"), BASES["b31"], BASES["b31"] + 10)
    cases = {}
    around = ["r:i:1", "ra:i:2", "rb:Z:x", "rcx:i:3", "rc0:i:4", "RC:Z:up", "rd:i:5", "q:i:6", "\x80c:i:7", "r\xff:i:8",
              "\xe9:Z:x", "a\x7f:i:9", "rc:Z:old"]
    for name, path in [("step", step), ("multi", multi), ("star", "*")]:
        cases["tags/around-rc/%s" % name] = rec(path, 9, 0, 9, tags=around)
        cases["tags/around-rc-rev/%s" % name] = rec(path, 9, 0, 9, tags=around[::-1])
        cases["tags/rc-only/%s" % name] = rec(path, 9, 0, 9, tags=["rc:Z:old"])
        cases["tags/no-rc/%s" % name] = rec(path, 9, 0, 9, tags=["ra:i:1", "rd:i:1"])
    many = ["t%02d:i:%d" % (i, i) for i in range(40)]
    for n in (15, 16, 17, 18):
        for name, path in [("step", step), ("multi", multi)]:
            body = many[:n - 1]   # + the cg tag rec() appends
            cases["tags/count-%d/%s" % (n, name)] = rec(path, 9, 0, 9, tags=body[::-1])
            cases["tags/count-%d-rc/%s" % (n, name)] = rec(path, 9, 0, 9, tags=body[:-1] + ["rc:Z:old"])
            for j in (0, n - 3, n - 2):   # a duplicate of the first field / of the last one collected / of the field after
                cases["tags/count-%d-dup%d/%s" % (n, j, name)] = rec(path, 9, 0, 9, tags=body + [body[j]])
            cases["tags/count-%d-dup-late/%s" % (n, name)] = rec(path, 9, 0, 9, tags=many[:n + 2] + [many[n + 1]])
    for n in (65528, 65529, 65530, 65531, 70000):
        v = "x" * (n - 5)
        cases["tags/field-%d" % n] = rec(step, 9, 0, 9, tags=["zz:Z:" + v, "aa:i:1"])
        cases["tags/field-%d-16" % n] = rec(step, 9, 0, 9, tags=many[:14] + ["zz:Z:" + v])
        cases["tags/field-%d-dup" % n] = rec(step, 9, 0, 9, tags=["zz:Z:" + v, "ab:i:2", "zz:i:1"])
    for n in (254, 255, 256, 300):
        k = "k" * n
        cases["tags/name-%d" % n] = rec(step, 9, 0, 9, tags=[k + ":i:1", "aa:i:1"])
        cases["tags/name-%d-dup" % n] = rec(step, 9, 0, 9, tags=[k + ":i:1", "aa:i:1", k + ":Z:2"])
        cases["tags/name-%d-prefix" % n] = rec(step, 9, 0, 9, tags=[k + ":i:1", k[:-1] + ":i:2"])
    for t in ["a:i", "ab:i", "ab::", "::::", "a::b", ":i:1", "ab:i:", "abcd", "ab:i:1:2", "rc:Z:", "rc:i:5"]:
        cases["tags/syntax/%r" % t] = rec(step, 9, 0, 9, tags=[t])
    cases["tags/empty-fields"] = rec(step, 9, 0, 9, tags=["", "zz:i:1", "", "aa:i:1", ""])
    return cases


def name_cases():
    """Contig names of 15, 16, 17 and 40 bytes, names that differ only in their last byte, chr1 next to chr10, SN
    prefixes id=...| (the lookup is by the whole SN; rc is the name without the prefix)."""
    cases = {}
    for k, sn in NAMES.items():
        cases["names/%s" % k] = rec(">%s:2-13" % sn, 11, 0, 11)
        cases["names/%s-bare" % k] = rec(sn, 16, 2, 13)
        cases["names/%s-rev" % k] = rec("<%s:8-16" % sn, 8, 0, 8)
        if len(sn) > 4:
            cases["names/%s-lastbyte" % k] = rec(">%s:2-13" % (sn[:-1] + "9"), 11, 0, 11)
            cases["names/%s-short" % k] = rec(">%s:2-13" % sn[:-1], 11, 0, 11)
            cases["names/%s-long" % k] = rec(">%s:2-13" % (sn + "1"), 11, 0, 11)
    cases["names/chr1-chr10"] = rec(">chr1:2-13>chr10:0-5", 16, 0, 16)
    cases["names/chr10-chr1"] = rec(">chr10:2-13>chr1:0-5", 16, 0, 16)
    cases["names/chr"] = rec(">chr:2-13", 11, 0, 11)
    cases["names/pfx-pfx2"] = rec(">id=HG7|chrP:2-13>id=HG8|chrP:0-5", 16, 0, 16)   # one reference contig chrP: no warning
    cases["names/pfx-stripped"] = rec(">chrP:2-13", 11, 0, 11)
    return cases


def path_cases():
    """Multi-contig warnings, an unknown contig, a bare name inside a multi-step path."""
    a, b = layout_contig("contiguous", "0"), layout_contig("gaps", "b53")
    b0 = 2**53
    cases = {
        "paths/warn-2": rec(">%s:3-12>%s:%d-%d" % (a, b, b0 + 20, b0 + 25), 14, 0, 14),
        "paths/warn-3": rec(">%s:3-12<%s:%d-%d>chr10:0-16" % (a, b, b0 + 20, b0 + 25), 30, 0, 30, tags=["rc:Z:old"]),
        "paths/warn-same-twice": rec(">%s:3-12>%s:0-5>%s:%d-%d" % (a, a, b, b0, b0 + 3), 17, 0, 17),
        "paths/warn-aligned": rec(">%s:0-10>%s:%d-%d" % (a, b, b0 + 20, b0 + 25), 15, 0, 15),   # whole nodes: gaf2paf converts it
        "paths/warn-aligned-3": rec("<%s:10-15>chr10:0-8>%s:%d-%d" % (a, b, b0 + 30, b0 + 38), 21, 0, 21),
        "paths/no-warn-same": rec(">%s:3-12<%s:0-5" % (a, a), 14, 0, 14),
        "paths/unknown": rec(">nosuch:0-5", 5, 0, 5),
        "paths/unknown-second": rec(">%s:3-12>nosuch:0-5" % a, 14, 0, 14),
        "paths/bare-unknown": rec("nosuch", 99, 0, 5),
        "paths/bare-in-multi": rec(">%s:3-12>%s" % (a, a), 14, 0, 14),
        "paths/bare-first-in-multi": rec(">%s>%s:3-12" % (a, a), 14, 0, 14),
        "paths/prefixed-bare-alone": rec(">%s" % a, 35, 3, 12),
        "paths/prefixed-bare-alone-rev": rec("<%s" % a, 35, 3, 12),
        "paths/node-name": rec(">s5", 10, 0, 5),
        "paths/empty-step": rec(">%s:3-12>" % a, 9, 0, 9),
        "paths/empty-first-step": rec("><%s:3-12" % a, 9, 0, 9),
        "paths/long": rec("".join(">%s:%d-%d" % (a, i % 30, i % 30 + 5) for i in range(300)), 1500, 0, 1500),
        "paths/long-multi": rec("".join(">%s:%d-%d" % (a if i % 7 else b, (i % 30) + (0 if i % 7 else b0), (i % 30) + 5 + (0 if i % 7 else b0)) for i in range(200)), 1000, 0, 1000),
    }
    return cases


def all_cases(g):
    cases = {}
    for part in (geometry_cases(g), text_cases(), tag_cases(), name_cases(), path_cases()):
        assert not set(part) & set(cases)
        cases.update(part)
    return cases


# rGFA syntax: each its own graph (and a few records on it)
def syntax_graphs():
    sp = ("S s1 AAAAAAAAAA LN:i:10 SN:Z:chrA SO:i:0 SR:i:0\nS s2 AAAAA LN:i:5 SN:Z:chrA SO:i:10 SR:i:0\n"
          "S\ts3\tAAAA\tSN:Z:chrB SO:i:0 SR:i:0\n")
    gfa2 = ("H\tVN:Z:2.0\nS\ts1\t10\tAAAAAAAAAA\tSN:Z:chrA\tSO:i:0\tSR:i:0\nS\ts2\t5\tAAAAA\tSN:Z:chrA\tSO:i:10\tSR:i:0\n"
            "S\ts3\t4\tAAAA\tSN:Z:chrB\tSO:i:0\tSR:i:0\nE\t*\ts1+\ts2+\t10$\t10$\t0\t0\t0M\n")
    eline = ("S\ts1\tAAAAAAAAAA\tSN:Z:chrA\tSO:i:0\tSR:i:0\nS\ts2\tAAAAA\tSN:Z:chrA\tSO:i:10\tSR:i:0\n"
             "S\ts3\tAAAA\tSN:Z:chrB\tSO:i:0\tSR:i:0\nE\t*\ts1+\ts2+\t10$\t10$\t0\t0\t0M\nL\ts1\t+\ts2\t+\t0M\n")
    sameid = ("S\ts1\tAAAAAAAAAA\tSN:Z:chrA\tSO:i:0\tSR:i:0\nS\ts01\tAAAAA\tSN:Z:chrA\tSO:i:10\tSR:i:0\n"
              "S\txs3\tAAAA\tSN:Z:chrB\tSO:i:0\tSR:i:0\nS\ts3\tAAA\tSN:Z:chrC\tSO:i:0\tSR:i:0\n")
    rank1 = ("S\ts1\tAAAAAAAAAA\tSN:Z:chrA\tSO:i:0\tSR:i:0\nS\ts2\tAAAAA\tSN:Z:chrA\tSO:i:10\tSR:i:0\n"
             "S\ts3\tAAAA\tSN:Z:chrB\tSO:i:0\tSR:i:0\nS\ts4\tAAAAAA\tSN:Z:alt\tSO:i:100\tSR:i:1\nL\ts1\t+\ts4\t+\t0M\n")
    recs = [rec(">chrA:0-15", 15, 0, 15), rec(">chrA:3-12<chrB:0-4", 13, 0, 13), rec("chrA", 15, 2, 14),
            rec(">chrB:1-3", 2, 0, 2), rec(">chrC:0-3", 3, 0, 3), rec(">alt:100-106>chrA:0-4", 10, 0, 10),
            rec(">alt:101-105", 4, 0, 4)]
    return {"spaces": sp, "gfa2": gfa2, "e-lines": eline, "same-id": sameid, "rank1": rank1}, recs


# ---- running and comparing ------------------------------------------------------------------------------------
def run(binary, args, env=None):
    p = subprocess.run([binary] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=dict(os.environ, **(env or {})))
    return (p.returncode if p.returncode >= 0 else 128 - p.returncode), p.stdout, p.stderr.decode("latin-1")


def warnings_of(err):
    """The multi-contig warnings in a stderr text (three lines each), without anything else the tool printed."""
    lines, out, i = err.split("\n"), [], 0
    while i < len(lines):
        if lines[i].startswith("[gaf2unstable] warning"):
            out += lines[i:i + 3]
            i += 3
        else:
            i += 1
    return "\n".join(out)


def same(ref, got, kind):
    """-> None when `got` (rc, stdout, stderr) is what the reference's `ref` asks, else the difference."""
    rrc, rout, rerr = ref
    rc, out, err = got
    if rrc == 139:   # a zero-length interval: the reference reads past an empty vector; the port and this library abort
        rrc = 134
    if rc != rrc:
        return "exit %d, reference %d" % (rc, rrc)
    if rc == 0 and out != rout:
        return "stdout differs"
    if rc != 0 and not (out == rout if kind == "port" else rout == out[:len(rout)]):
        return "stdout is not the reference's (prefix)"
    if rc in (0, 134) and warnings_of(err) != warnings_of(rerr):
        return "warnings differ"
    if rc == 0 and err != rerr:
        return "stderr differs"
    return None


@pytest.fixture(scope="module")
def table():
    g = main_graph()
    cases = all_cases(g)
    ref, kind = H.oracle_path("auto", "gaf2unstable")
    td = tempfile.TemporaryDirectory()
    gp = os.path.join(td.name, "g.gfa")
    open(gp, "wb").write(g.text())
    files = {}
    for i, (name, line) in enumerate(cases.items()):
        p = os.path.join(td.name, "c%d.gaf" % i)
        open(p, "wb").write(("\n".join([ordinary(i), line, ordinary(i + 1)]) + "\n").encode("latin-1"))
        files[name] = p
    refs = dict(zip(files, POOL.map(lambda n: run(ref, [files[n], "-g", gp]), files)))
    yield {"graph": g, "gp": gp, "cases": cases, "files": files, "refs": refs, "kind": kind, "ref": ref, "dir": td.name}
    td.cleanup()


def test_table_reaches_every_outcome(table):
    """The table holds records the reference converts, warns on and aborts on, in every part, and zero-length
    intervals; the geometry covers every layout at every base both ways."""
    refs = table["refs"]
    for part in ("geo", "text", "tags", "names", "paths"):
        rcs = {refs[n][0] for n in refs if n.startswith(part + "/")}
        assert 0 in rcs and 134 in rcs, part
    assert sum(1 for n in refs if refs[n][0] == 0 and "warning" in refs[n][2]) >= 15
    tags = [n for n in refs if n.startswith("tags/")]
    assert sum(1 for n in tags if refs[n][0] == 0) > len(tags) // 2
    for bk in BASES:
        for lay in LAYOUTS:
            got = [refs[n][0] for n in refs if n.startswith("geo/%s/%s/" % (lay, bk))]
            assert got.count(0) >= 3 and len(got) - got.count(0) >= 3, (lay, bk)
    assert len(table["cases"]) > 2000


@pytest.mark.parametrize("runner", sorted(RUNNERS))
def test_each_case_alone(table, runner):
    binary, env = RUNNERS[runner]
    gp, files, refs = table["gp"], table["files"], table["refs"]
    got = dict(zip(files, POOL.map(lambda n: run(binary, [files[n], "-g", gp], env), files)))
    bad = {n: d for n in files for d in [same(refs[n], got[n], table["kind"])] if d}
    assert not bad, "%d of %d cases differ, e.g. %s" % (len(bad), len(files), sorted(bad.items())[:8])


def combined(table, seed):
    """The cases the reference does not abort on, in a seeded order, with ordinary records in between."""
    rnd = random.Random(seed)
    names = [n for n in table["files"] if table["refs"][n][0] == 0]
    rnd.shuffle(names)
    lines = []
    for i, n in enumerate(names):
        lines.append(table["cases"][n])
        if i % 3 == 0:
            lines.append(ordinary(i))
    return ("\n".join(lines) + "\n").encode("latin-1")


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_all_cases_together(table, seed):
    """One input of every non-aborting case: per runner, the exit code, stdout, the warnings verbatim and the -o file."""
    data = combined(table, seed)
    d = table["dir"]
    ap, lp = os.path.join(d, "all%d.gaf" % seed), os.path.join(d, "all%d.tsv" % seed)
    open(ap, "wb").write(data)
    ref = run(table["ref"], [ap, "-g", table["gp"], "-o", lp])
    ref_nl = open(lp, "rb").read()
    assert ref[0] == 0 and ref[2].count("[gaf2unstable] warning") >= 4
    for runner, (binary, env) in sorted(RUNNERS.items()):
        os.remove(lp)
        got = run(binary, [ap, "-g", table["gp"], "-o", lp], env)
        assert got == ref, runner
        assert open(lp, "rb").read() == ref_nl, runner


def test_emulator_takes_several_stride_turns(table):
    """k_unstable under the emulator loops over the records: the combined input takes more than one turn of its grid."""
    data = combined(table, 1)
    p = subprocess.run([SIMT, "-g", table["gp"], "-"], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       env=dict(os.environ, G2P_SIMT_STATS="1"))
    stats = [ln for ln in p.stderr.decode("latin-1").split("\n") if ln.startswith("g2u_simt:")]
    assert p.returncode == 0 and stats and stats[0].startswith("g2u_simt: k_unstable, ")
    turns = int(stats[0].split(" stride turns")[0].rsplit(" ", 1)[1])
    assert turns > 4, stats


def test_warning_then_abort(table):
    """Warnings for records before a record the reference aborts on are printed; none after it."""
    cases = table["cases"]
    w = cases["paths/warn-2"]
    data = "\n".join([ordinary(0), w, ordinary(1), cases["paths/warn-3"], cases["paths/unknown"], w, ordinary(2)]) + "\n"
    d = table["dir"]
    ap = os.path.join(d, "warn-abort.gaf")
    open(ap, "wb").write(data.encode())
    ref = run(table["ref"], [ap, "-g", table["gp"]])
    assert ref[0] == 134 and warnings_of(ref[2]).count("[gaf2unstable] warning") == 2
    for runner, (binary, env) in sorted(RUNNERS.items()):
        assert same(ref, run(binary, [ap, "-g", table["gp"]], env), table["kind"]) is None, runner


@pytest.mark.parametrize("name", sorted(syntax_graphs()[0]))
def test_rgfa_syntax(name):
    graphs, recs = syntax_graphs()
    ref, kind = H.oracle_path("auto", "gaf2unstable")
    with tempfile.TemporaryDirectory() as td:
        gp, lp = os.path.join(td, "g.gfa"), os.path.join(td, "l.tsv")
        open(gp, "w").write(graphs[name])
        outcomes = set()
        for i, r in enumerate(recs):
            ap = os.path.join(td, "a%d.gaf" % i)
            open(ap, "w").write(r + "\n" + recs[0] + "\n")
            want = run(ref, [ap, "-g", gp, "-o", lp])
            nl = open(lp, "rb").read() if want[0] == 0 else None
            outcomes.add(want[0])
            for runner, (binary, env) in sorted(RUNNERS.items()):
                if os.path.exists(lp):
                    os.remove(lp)
                got = run(binary, [ap, "-g", gp, "-o", lp], env)
                assert same(want, got, kind) is None, (runner, r, got, want)
                if nl is not None:
                    assert open(lp, "rb").read() == nl, runner
        assert 0 in outcomes


# ---- GPU ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_each_case_and_the_executable(g2p, table):
    """Converter.unstable_host on each case alone and on the combined inputs; bin/gaf2unstable on the combined inputs
    and on the aborting cases of the path and tag parts."""
    exe = os.path.join(g2p.BIN_DIR, "gaf2unstable")
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(table["graph"].text())
        assert ok
        bad = {}
        for name, path in table["files"].items():
            data = open(path, "rb").read()
            out, res, warns = cv.unstable_host(data)
            rc = g2p.exit_code(res)
            d = same(table["refs"][name], (rc, out, "".join(warns)), table["kind"])
            if d:
                bad[name] = d
        assert not bad, "%d cases differ, e.g. %s" % (len(bad), sorted(bad.items())[:8])
        for seed in (1, 2, 3):
            data = combined(table, seed)
            ap, lp, lp2 = (os.path.join(table["dir"], x) for x in ("gpu%d.gaf" % seed, "gpu%d.tsv" % seed, "gpu%d_ref.tsv" % seed))
            open(ap, "wb").write(data)
            ref = run(table["ref"], [ap, "-g", table["gp"], "-o", lp2])
            out, res, warns = cv.unstable_host(data)
            assert (g2p.exit_code(res), out, "".join(warns)) == ref
            assert run(exe, [ap, "-g", table["gp"], "-o", lp]) == ref
            assert open(lp, "rb").read() == open(lp2, "rb").read() == cv.node_lengths()
        aborts = [n for n in table["files"] if n.startswith(("paths/", "tags/")) and table["refs"][n][0] != 0]
        assert aborts
        for n in aborts:
            assert same(table["refs"][n], run(exe, [table["files"][n], "-g", table["gp"]]), table["kind"]) is None, n
    finally:
        cv.close()


def fused_reference(table, data):
    """`gaf2unstable | gaf2paf -l <its -o file>` of the checkers -> (stage-1 (rc, out, err), stage-2 (rc, out, err), the
    record of the intermediate GAF at which stage 2 stops, or None)."""
    ref2, _k = H.oracle_path("auto", "gaf2paf")
    with tempfile.TemporaryDirectory() as td:
        ap, lp, mp = (os.path.join(td, x) for x in ("a.gaf", "l.tsv", "m.gaf"))
        open(ap, "wb").write(data)
        r1 = run(table["ref"], [ap, "-g", table["gp"], "-o", lp])
        open(mp, "wb").write(r1[1])
        r2 = run(ref2, [mp, "-l", lp])
        stop = None
        if r2[0] != 0:   # the first record whose prefix of the intermediate fails
            mid = r1[1].split(b"\n")[:-1]
            for k in range(len(mid)):
                open(mp, "wb").write(b"\n".join(mid[:k + 1]) + b"\n")
                if run(ref2, [mp, "-l", lp])[0] != 0:
                    stop = k
                    break
    return r1, r2, stop


@pytest.mark.gpu
def test_gpu_fused_call_matches_the_two_checkers(g2p, table):
    """unstable_convert_host on each case alone against the checkers' two processes: the PAF, which stage stopped
    (res.stage) and at which record (err_record), and the stage-1 warning text."""
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(table["graph"].text())
        assert ok
        bad, stages = {}, set()
        for name, path in table["files"].items():
            data = open(path, "rb").read()
            (rc1, out1, err1), (rc2, out2, err2), stop = fused_reference(table, data)
            paf, res, warn_text = cv.unstable_convert_host(data)
            if rc2 != 0:          # gaf2paf stops on the intermediate (what stage 1 wrote before it stopped, if it did)
                want = (2, stop, 1 if rc2 == 1 else 134)
            elif rc1 != 0:        # stage 1 stops at the case, the record between two ordinary ones
                want = (1, 1, 134)
            else:
                want = (0, None, 0)
            stages.add(want[0])
            got = (res.stage, res.err_record if want[1] is not None else None, g2p.exit_code(res))
            if got != want:
                bad[name] = "stage / record / exit %r, reference %r" % (got, want)
            elif not (paf == out2 if rc2 in (0, 1) or table["kind"] == "port" else out2 == paf[:len(out2)]):
                bad[name] = "paf differs"
            elif warnings_of(warn_text) != warnings_of(err1) or (rc1 == 0 and warn_text != err1):
                bad[name] = "warnings differ"
        assert not bad, "%d cases differ, e.g. %s" % (len(bad), sorted(bad.items())[:8])
        assert stages == {0, 1, 2}
    finally:
        cv.close()


# ---- output past 4 GiB --------------------------------------------------------------------------------------
# 10 000 records of about 60 bytes, each spanning a contig of 65 536 one-base nodes: about 448 kB of output per record,
# 4.48 GB in all -- more than the fused call's gaf2paf stage (< 4 GiB of input) can take.
WIDE_NODES, WIDE_RECORDS = 65536, 10000


def wide_graph():
    lines = ["S\ts%d\tA\tLN:i:1\tSN:Z:W\tSO:i:%d\tSR:i:0" % (i + 1, i) for i in range(WIDE_NODES)]
    return ("\n".join(lines) + "\n").encode()


def wide_record():
    return ("q\t%d\t0\t%d\t+\t>W:0-%d\t%d\t0\t%d\t%d\t%d\t60\tcg:Z:%dM\n" % ((WIDE_NODES,) * 8)).encode()


@pytest.mark.gpu
def test_gpu_fused_call_refuses_an_intermediate_of_4gib(g2p):
    """The fused call's gaf2paf stage takes less than 4 GiB: an intermediate GAF of 4.48 GB made from 700 kB of input is
    refused with G2P_E_TOOBIG before that stage runs."""
    import time
    import torch
    rgfa, one = wide_graph(), wide_record()
    free0 = torch.cuda.mem_get_info()[0]
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(rgfa)
        assert ok
        t0 = time.perf_counter()
        with pytest.raises(g2p.G2PError, match="error %d:" % g2p.G2P_E_TOOBIG):
            cv.unstable_convert_host(one * WIDE_RECORDS)
        print("\n[measure] fused call refusing %d records: %.2f s, device memory held by the context %.2f GB"
              % (WIDE_RECORDS, time.perf_counter() - t0, (free0 - torch.cuda.mem_get_info()[0]) / 1e9))
        out, res, warns = cv.unstable_host(one)
        assert g2p.exit_code(res) == 0 and len(out) * WIDE_RECORDS >= 2**32   # the intermediate passes 4 GiB
        # also when stage 1 stops at a record after the first 4 GiB of its output
        bad = one * WIDE_RECORDS + b"q\t5\t0\t5\t+\t>nosuch:0-5\t5\t0\t5\t5\t5\t60\n" + one
        with pytest.raises(g2p.G2PError, match="error %d:" % g2p.G2P_E_TOOBIG):
            cv.unstable_convert_host(bad)
        # and the context still converts afterwards
        paf, res, warn_text = cv.unstable_convert_host(one * 3)
        assert g2p.exit_code(res) == 0 and res.mid_bytes == 3 * len(out) and warn_text == ""
        assert paf and paf == H.run_gaf2paf_cpu(out * 3, cv.node_lengths())[1]
    finally:
        cv.close()


@pytest.mark.gpu
def test_gpu_unstable_host_output_past_4gib(g2p):
    """One g2p_unstable_host call whose output is 4.48 GB (u64 offsets in k_unstable and in the scans), and the same
    input through bin/gaf2unstable: N copies of the checker's output for one record, hashed as it streams."""
    import ctypes
    import time
    import torch
    rgfa, one = wide_graph(), wide_record()
    ref, kind = H.oracle_path("auto", "gaf2unstable")
    with tempfile.TemporaryDirectory() as td:
        gp, ap = os.path.join(td, "g.gfa"), os.path.join(td, "a.gaf")
        open(gp, "wb").write(rgfa)
        open(ap, "wb").write(one)
        rc, ref_one, err = run(ref, [ap, "-g", gp])
        assert rc == 0 and len(ref_one) * WIDE_RECORDS > 2**32
        want = hashlib.sha256()
        for _ in range(WIDE_RECORDS):
            want.update(ref_one)
        want = want.hexdigest()

        def digest(addr, n):
            h, step = hashlib.sha256(), 1 << 28
            for a in range(0, n, step):
                h.update((ctypes.c_char * min(step, n - a)).from_address(addr + a))
            return h.hexdigest()

        cv = g2p.Converter(0)
        try:
            ok, code, msg = cv.load_rgfa(rgfa)
            assert ok
            data = one * WIDE_RECORDS
            addr, n, keep = g2p._buf_ptr(data)
            out, res = ctypes.c_void_p(), g2p.Result()
            free0 = torch.cuda.mem_get_info()[0]
            t0 = time.perf_counter()
            assert g2p.lib.g2p_unstable_host(cv._h, addr, n, ctypes.byref(out), ctypes.byref(res)) == g2p.G2P_OK
            print("\n[measure] g2p_unstable_host, %d bytes in, %d bytes out: %.2f s (device %.1f ms), device memory held by "
                  "the context %.2f GB" % (n, res.out_bytes, time.perf_counter() - t0, res.device_ms, (free0 - torch.cuda.mem_get_info()[0]) / 1e9))
            assert g2p.exit_code(res) == 0 and res.n_records == WIDE_RECORDS
            assert res.out_bytes == len(ref_one) * WIDE_RECORDS
            assert digest(out.value, res.out_bytes) == want
        finally:
            cv.close()
        big = os.path.join(td, "big.gaf")
        open(big, "wb").write(one * WIDE_RECORDS)
        t0 = time.perf_counter()
        p = subprocess.Popen([os.path.join(g2p.BIN_DIR, "gaf2unstable"), big, "-g", gp], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        h, n = hashlib.sha256(), 0
        while True:
            b = p.stdout.read(1 << 24)
            if not b:
                break
            h.update(b)
            n += len(b)
        err = p.stderr.read()
        assert p.wait() == 0, err
        print("[measure] bin/gaf2unstable, %d bytes out, read and hashed: %.2f s" % (n, time.perf_counter() - t0))
        assert n == len(ref_one) * WIDE_RECORDS and h.hexdigest() == want


@pytest.mark.gpu
def test_gpu_fused_warnings_survive_a_later_unstable_call(g2p, table):
    """g2p_unstable_convert_warnings gives the warnings of the last fused call, also after a g2p_unstable_host call on
    the same context with warnings of its own."""
    import torch
    cases = table["cases"]
    a = ("\n".join([ordinary(0), cases["paths/warn-aligned"], ordinary(1), cases["paths/warn-aligned-3"]]) + "\n").encode("latin-1")
    b = ("\n".join([cases["paths/warn-same-twice"], ordinary(2), ordinary(3), cases["tags/around-rc/multi"], cases["paths/warn-2"]]) + "\n").encode("latin-1")
    (rc1, out1, err_a), (rc2, paf_a, _e), _stop = fused_reference(table, a)
    with tempfile.TemporaryDirectory() as td:
        bp = os.path.join(td, "b.gaf")
        open(bp, "wb").write(b)
        rb = run(table["ref"], [bp, "-g", table["gp"]])
    assert rc1 == rc2 == 0 and rb[0] == 0
    assert err_a.count("[gaf2unstable] warning") == 2 and rb[2].count("[gaf2unstable] warning") == 3
    cv = g2p.Converter(0)
    try:
        ok, code, msg = cv.load_rgfa(table["graph"].text())
        assert ok
        t = torch.empty(len(a) + 16, dtype=torch.uint8, device="cuda")
        g2p.copy_to_device(t.data_ptr(), a)
        torch.cuda.synchronize()
        d_out, res = cv.unstable_convert_device(t.data_ptr(), len(a), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert g2p.exit_code(res) == 0 and g2p.copy_to_host(d_out, res.out_bytes) == paf_a
        out, res_b, warns = cv.unstable_host(b)
        assert out == rb[1] and "".join(warns) == rb[2]
        assert cv._convert_warnings() == err_a
        assert cv._convert_warnings() == err_a
    finally:
        cv.close()
