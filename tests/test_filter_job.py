"""gaffilter on inputs of any size and on several GPUs: the filter job (g2p_filter_job_*, csrc/g2p_filter_job.hpp), which
partitions the records by query name.  Its results must equal the single g2p_filter_host call on every input that call
accepts: exit code, stdout bytes, stderr.  CPU tests run the job's three passes under the SIMT emulator
(build/g2p_filter_job_simt -c BYTES -P PARTS, compared with the single call under build/g2p_filter_simt) and its
partition planner (--plan); the GPU tests go through FilterJob and the
gaffilter executable, including inputs beyond the single call's 4 GiB."""
import hashlib
import os
import re
import shutil
import subprocess
import tempfile

import pytest

import helpers as H
from test_filter import EDGE_BAD, EDGE_GAF, OPTION_SETS, QUIRKS, assert_partial, last_line, ref_gaffilter, simt

JOB_SIMT = os.path.join(H.BUILD, "g2p_filter_job_simt")
CHUNKINGS = [(200, 1), (4096, 3), (65536, 256)]
# (the emulator takes ~0.1 s per chunk: 200-byte chunks get inputs of a few KB)


@pytest.fixture(scope="module", autouse=True)
def _job_simt():
    if not os.path.exists(JOB_SIMT):
        subprocess.check_call(["make", "-C", H.ROOT, JOB_SIMT[len(H.ROOT) + 1:]], stdout=subprocess.DEVNULL)


def job_simt(text, args):
    p = subprocess.run([JOB_SIMT] + args + ["-"], input=text, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return p.returncode, p.stdout, p.stderr.decode("latin-1")


def same_chunked(text, args, chunkings=CHUNKINGS, partial=True):
    """The job under the emulator, for every (chunk bytes, partitions) of `chunkings`, equals the unchunked emulator run and
    the checker: exit code, stdout bytes, summary line."""
    rc, out, err = simt(text, args)
    crc, cout, cerr = ref_gaffilter(text, args)
    assert (rc, out) == (crc, cout), (args, rc, crc, err[-300:])
    if rc == 0:
        assert last_line(err) == last_line(cerr), args
        if partial:
            assert_partial(err, args)
    for c, parts in chunkings:
        jrc, jout, jerr = job_simt(text, args + ["-c", str(c), "-P", str(parts)])
        assert (jrc, jout) == (rc, out), (args, c, parts, jerr[-300:])
        assert last_line(jerr) == last_line(err), (args, c, parts)
    return rc, out, err


@pytest.mark.parametrize("paf", [False, True])
def test_emulated_job_matches_single_call(paf):
    text, _ = H.gen_filter_case(41, n_records=400, n_queries=70, paf=paf)
    small, _ = H.gen_filter_case(42, n_records=40, n_queries=6, paf=paf)
    for args in OPTION_SETS:
        a = args + (["-p"] if paf else [])
        same_chunked(text, a, chunkings=CHUNKINGS[1:])
        same_chunked(small, a, chunkings=CHUNKINGS[:1])


def test_emulated_job_spread_queries():
    """Three queries whose overlaps cross many chunks and partitions (each query's rows come from every chunk)."""
    text = H.gen_spread_filter_case(78, n_records=1000, n_queries=3)
    for args in (["-r", "2"], ["-o", "300"]):
        same_chunked(text, args, chunkings=[(8192, 1), (16384, 3), (32768, 256)])


def test_emulated_job_edges():
    # an unterminated last line; more partitions than non-empty buckets (three queries, 256 partitions)
    assert not EDGE_GAF.endswith(b"\n")
    for args in (["-r", "2"], ["-o", "5"]):
        same_chunked(EDGE_GAF, args, chunkings=[(1, 1), (150, 256), (1 << 20, 256)], partial=False)
    # chunks that hold no loaded line (only '*' lines)
    base, _ = H.gen_filter_case(43, n_records=60, n_queries=8)
    lines = base.split(b"\n")[:-1]
    stars = b"*\t>s43\t97\t12\t0\t6\t92\n" * 40
    text = b"\n".join(lines[:30]) + b"\n" + stars + b"\n".join(lines[30:]) + b"\n" + stars
    same_chunked(text, ["-r", "2"], chunkings=[(300, 3), (700, 256)])
    # the signed 64-bit sum of the filtered block lengths wraps the same way when it is summed over partitions
    data, args = QUIRKS[6]
    extra = data.replace(b"q1\t", b"q7\t").replace(b"q2\t", b"q8\t")
    rc, out, err = same_chunked(data + extra, args, chunkings=[(60, 256), (200, 3)], partial=False)
    assert rc == 0 and int(last_line(err).split()[-1]) < 0


def abort_line(err):
    m = re.search(r"abort: (?:line|assertion of the filter loop on record) (\d+)", err)
    assert m, err
    return int(m.group(1))


def test_emulated_job_error_precedence():
    base, _ = H.gen_filter_case(44, n_records=50, n_queries=8)
    # a parse error in a late chunk wins over an assertion pair in an early one: 134, nothing printed, the parse
    # error's global line
    assertion = QUIRKS[0][0]
    bad = EDGE_BAD[0][0]
    text = assertion + base + bad
    bad_line = (assertion + base).count(b"\n") + bad.split(b"\n").index(next(ln for ln in bad.split(b"\n") if b"q2\t\t0" in ln))
    rc, out, err = simt(text, ["-r", "2"])
    assert rc == 134 and out == b"" and abort_line(err) == bad_line and "abort: line" in err
    for c, parts in CHUNKINGS:
        jrc, jout, jerr = job_simt(text, ["-r", "2", "-c", str(c), "-P", str(parts)])
        assert (jrc, jout, last_line(jerr)) == (134, b"", last_line(err)), (c, parts)
    # assertion pairs of several queries (in several partitions): the smallest global line
    pairs = b"".join(QUIRKS[0][0].replace(b"q1\t", b"z%d\t" % k).replace(b"q2\t", b"y%d\t" % k) for k in range(8))
    text = base + pairs
    rc, out, err = simt(text, ["-r", "2"])
    assert rc == 134 and out == b""
    assert abort_line(err) >= base.count(b"\n")
    for c, parts in CHUNKINGS:
        jrc, jout, jerr = job_simt(text, ["-r", "2", "-c", str(c), "-P", str(parts)])
        assert (jrc, jout, last_line(jerr)) == (134, b"", last_line(err)), (c, parts)
    # a query_start >= 2^32 - 16 in a late chunk: the single call's error
    huge = b"q5\t99999999999\t4294967290\t4294967299\t+\t>a\t50\t0\t9\t9\t9\t60\n"
    text = base + huge
    rc, out, err = simt(text, ["-r", "2"])
    assert rc == 98 and out == b""
    for c, parts in CHUNKINGS:
        assert job_simt(text, ["-r", "2", "-c", str(c), "-P", str(parts)])[:2] == (98, b"")


def plan(rows, cap, min_parts, ngpu):
    p = subprocess.run([JOB_SIMT, "--plan", str(cap), str(min_parts), str(ngpu)], input=" ".join(map(str, rows)).encode(),
                       stdout=subprocess.PIPE)
    if p.returncode:
        return p.returncode, p.stdout.decode()
    return 0, [tuple(int(x) for x in ln.split()) for ln in p.stdout.decode().split("\n") if ln]


def check_plan(rows, cap, min_parts, ngpu):
    rc, parts = plan(rows, cap, min_parts, ngpu)
    assert rc == 0, parts
    # contiguous bucket ranges covering 0..256, row counts summed correctly, each within the capacity
    assert parts[0][0] == 0 and parts[-1][1] == 256
    for (a0, a1, _, _), (b0, _, _, _) in zip(parts, parts[1:]):
        assert a1 == b0 and a0 < a1
    for b0, b1, r, g in parts:
        assert r == sum(rows[b0:b1]) and r <= cap and 0 <= g < ngpu
    assert len(parts) >= min(256, max(min_parts, ngpu, -(-sum(rows) // cap)))
    return parts


def test_partition_planner():
    import random
    rnd = random.Random(5)
    assert check_plan([0] * 256, 100, 1, 1) == [(0, 256, 0, 0)]
    parts = check_plan([0] * 256, 100, 256, 1)   # more partitions than non-empty buckets
    assert len(parts) == 256
    rows = [rnd.randrange(1000) for _ in range(256)]
    for cap, min_parts, ngpu in ((10 ** 9, 1, 1), (10 ** 9, 5, 2), (3000, 1, 1), (1000, 1, 8), (10 ** 9, 300, 3)):
        parts = check_plan(rows, cap, min_parts, ngpu)
        if ngpu > 1:   # balanced over the GPUs by row count
            load = [sum(r for _, _, r, g in parts if g == k) for k in range(ngpu)]
            assert max(load) - min(load) <= max(r for _, _, r, _ in parts)
    skew = [0] * 256
    skew[7], skew[200] = 5000, 3
    parts = check_plan(skew, 5000, 4, 2)
    assert any(r == 5000 for _, _, r, _ in parts)
    # one bucket beyond a GPU's capacity (a single query with that many alignments): no plan
    rc, msg = plan(skew, 4999, 1, 1)
    assert rc == 3 and "single query sequence" in msg


# ---- on the GPU ------------------------------------------------------------------------------------------------------
def n_gpus():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout
        return sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
    except Exception:
        return 0


def pieces(text, size):
    """newline-aligned chunks of about `size` bytes"""
    out, pos = [], 0
    while pos < len(text):
        end = min(len(text), pos + size)
        if end < len(text):
            nl = text.rfind(b"\n", pos, end)
            if nl >= 0:
                end = nl + 1
            else:
                q = text.find(b"\n", end)
                end = len(text) if q < 0 else q + 1
        out.append(text[pos:end])
        pos = end
    return out


def run_job(g2p, cvs, params, chunks):
    job = g2p.FilterJob(cvs, params)
    try:
        for c, t in enumerate(chunks):
            job.load(c, t)
        res = job.decide()
        if res.rec_status:
            return res, None
        return res, b"".join(job.emit(c, t)[0] for c, t in enumerate(chunks))
    finally:
        job.close()


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [1, 2])
@pytest.mark.parametrize("paf", [False, True])
def test_gpu_filter_job_matches_single_call(g2p, monkeypatch, gpus, paf):
    if n_gpus() < gpus:
        pytest.skip("needs %d GPUs" % gpus)
    monkeypatch.setenv("G2P_FILTER_PARTS", "7")
    text, _ = H.gen_filter_case(21, 60000, 4000, paf)
    cvs = [g2p.Converter(g) for g in range(gpus)]
    try:
        for args, kw in ((["-r", "2"], dict(ratio=2)), (["-o", "150", "-b", "60"], dict(min_overlap_length=150, min_block_length=60))):
            params = g2p.Converter.filter_params(paf=paf, **kw)
            out, res = cvs[0].filter_host(text, params)
            jres, jout = run_job(g2p, cvs, params, pieces(text, 100000))
            assert jout == out
            for f in ("n_loaded", "n_filtered", "filtered_len", "rec_status", "err_record"):
                assert getattr(jres, f) == getattr(res, f), f
            crc, cout, cerr = ref_gaffilter(text, args + (["-p"] if paf else []))
            assert crc == 0 and cout == out
            assert_partial(cerr)
        # abort cases: an assertion pair, then a parse error after it
        for bad in (QUIRKS[0][0], QUIRKS[0][0] + EDGE_BAD[0][0]):
            data = text[:text.rfind(b"\n", 0, 300000) + 1] + bad if not paf else None
            if data is None:
                continue
            params = g2p.Converter.filter_params(ratio=2)
            out, res = cvs[0].filter_host(data, params)
            jres, jout = run_job(g2p, cvs, params, pieces(data, 30000))
            assert res.rec_status >= 16 and (jres.rec_status, jres.err_record) == (res.rec_status, res.err_record) and jout is None
    finally:
        for cv in cvs:
            cv.close()


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [1, 2])
def test_gpu_gaffilter_cli_job_matches_single_call(g2p, gpus):
    if n_gpus() < gpus:
        pytest.skip("needs %d GPUs" % gpus)
    exe = os.path.join(g2p.BIN_DIR, "gaffilter")
    text, _ = H.gen_filter_case(31, 20000, 900, False)
    cut1, cut2 = text.rfind(b"\n", 0, 200000) + 1, text.rfind(b"\n", 0, 400000) + 1
    bad = text[:cut1] + QUIRKS[0][0] + text[cut1:cut2]
    worse = bad + EDGE_BAD[0][0]
    env = dict(os.environ, G2P_GPUS=str(gpus), G2P_CHUNK_BYTES="65536", G2P_FILTER_PARTS="5", G2P_IO_MIN_BYTES="16384")
    with tempfile.TemporaryDirectory() as td:
        for data, args in ((text, ["-r", "2"]), (text, ["-o", "100"]), (bad, ["-r", "2"]), (worse, ["-r", "2"])):
            gp = os.path.join(td, "in.gaf")
            open(gp, "wb").write(data)
            single = subprocess.run([exe] + args + [gp], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            if data is text:
                assert single.returncode == 0
                assert_partial(single.stderr.decode())
            else:
                assert single.returncode != 0 and single.stdout == b""
            for src in ("file", "stdin"):
                for sink in ("pipe", "file"):
                    op = os.path.join(td, "out")
                    with open(op, "wb") as of:
                        p = subprocess.run([exe] + args + [gp if src == "file" else "-"], input=None if src == "file" else data, env=env,
                                           stdout=subprocess.PIPE if sink == "pipe" else of, stderr=subprocess.PIPE)
                    out = p.stdout if sink == "pipe" else open(op, "rb").read()
                    assert (p.returncode, out, p.stderr) == (single.returncode, single.stdout, single.stderr), (args, src, sink, p.stderr[-300:])


BASE_CASE = (61, 60000, 4000, False)


def renamed(text, k):
    """the records of `text` with their query names prefixed c{k}_ ('*' lines unchanged)"""
    pre = b"c%d_" % k
    t = text.replace(b"\nq", b"\n" + pre + b"q")
    return pre + t if t.startswith(b"q") else t


@pytest.mark.gpu
def test_gpu_filter_job_beyond_4gib(g2p):
    """K renamed copies of a 60 000-record base, more than 4 GiB in all, through FilterJob chunk by chunk (the input is
    never materialised): each chunk prints the base's kept records under its prefix, the totals are K times the base's."""
    base, _ = H.gen_filter_case(*BASE_CASE)
    cv = g2p.Converter(0)
    try:
        params = g2p.Converter.filter_params(ratio=2)
        bout, bres = cv.filter_host(base, params)
        assert bres.rec_status == 0 and 0 < bres.n_filtered < bres.n_loaded
        K = (4 << 30) // len(base) + 2
        assert K * len(base) > 0xFFFFFFF0
        job = g2p.FilterJob([cv], params)
        try:
            for k in range(K):
                job.load(k, renamed(base, k))
            res = job.decide()
            assert res.rec_status == 0
            assert (res.n_loaded, res.n_filtered, res.filtered_len) == (K * bres.n_loaded, K * bres.n_filtered, (K * bres.filtered_len) % (1 << 64))
            for k in range(K):
                out, r = job.emit(k, renamed(base, k))
                assert out == renamed(bout, k), k
        finally:
            job.close()
    finally:
        cv.close()


@pytest.mark.gpu
def test_gpu_gaffilter_cli_beyond_4gib(g2p):
    """The same input as a > 4 GiB file through the gaffilter executable: md5 of the streamed stdout, the summary."""
    exe = os.path.join(g2p.BIN_DIR, "gaffilter")
    base, _ = H.gen_filter_case(*BASE_CASE)
    K = (4 << 30) // len(base) + 2
    td = tempfile.mkdtemp()
    try:
        if shutil.disk_usage(td).free < K * len(base) + (2 << 30):
            pytest.skip("the temporary directory has less than %d bytes free for the > 4 GiB input" % (K * len(base) + (2 << 30)))
        cv = g2p.Converter(0)
        try:
            bout, bres = cv.filter_host(base, g2p.Converter.filter_params(ratio=2))
        finally:
            cv.close()
        gp = os.path.join(td, "big.gaf")
        want = hashlib.md5()
        with open(gp, "wb") as f:
            for k in range(K):
                f.write(renamed(base, k))
                want.update(renamed(bout, k))
        p = subprocess.Popen([exe, "-r", "2", gp], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        got = hashlib.md5()
        while True:
            b = p.stdout.read(1 << 22)
            if not b:
                break
            got.update(b)
        err = p.stderr.read().decode()
        assert p.wait() == 0, err[-500:]
        assert got.hexdigest() == want.hexdigest()
        assert last_line(err) == "[gaffilter]: filtered %d / %d. total block lengths filtered: %d" % (K * bres.n_filtered, K * bres.n_loaded, K * bres.filtered_len)
    finally:
        shutil.rmtree(td, ignore_errors=True)
