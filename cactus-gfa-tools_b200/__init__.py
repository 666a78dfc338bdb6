"""cactus-gfa-tools_b200 — B200-native GAF -> PAF conversion (gaf2paf / gaf2unstable path).

Thin ctypes binding over the C-ABI of ``lib/libg2p.so`` (``include/g2p.h``).  The
reference (ComparativeGenomicsToolkit/cactus-gfa-tools) exposes this path only as the
``gaf2paf`` / ``gaf2unstable`` executables; the functions here mirror those two command
lines (``gaf2paf(gaf, lengths)`` ~ ``gaf2paf -l lengths.tsv in.gaf``) so that parity
tests read like the reference's ``test/gaf2paf.t``.

There is no CPU fallback: importing works anywhere (so that CPU-only CI can check the
exported symbols), but creating a :class:`Converter` without a CUDA device raises
:class:`G2PError`, and a missing ``libg2p.so`` raises at import.

The directory name contains a hyphen (it is the name the build contract fixes), so
import it through the ``cactus_gfa_tools_b200`` shim module at the repository root.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libg2p.so")
BIN_DIR = os.path.join(_HERE, "bin")

# include/g2p.h
G2P_OK = 0
G2P_E_NO_DEVICE = -1
G2P_E_CUDA = -2
G2P_E_ARG = -3
G2P_E_TABLE = -4
G2P_E_NOTABLE = -5
G2P_E_TOOBIG = -6

REC_OK = 0
REC_ERR_NAME = 1
REC_ERR_NOCG = 2
REC_ABORT = 16

EXPORTED_SYMBOLS = (
    "g2p_create", "g2p_destroy", "g2p_last_error", "g2p_host_alloc", "g2p_host_free", "g2p_load_lengths",
    "g2p_table_entries", "g2p_copy_to_device", "g2p_copy_to_host", "g2p_convert_device", "g2p_convert_host", "g2p_index_lines", "g2p_format_error",
    "g2p_load_rgfa", "g2p_share_rgfa", "g2p_rgfa_node_lengths", "g2p_unstable_device", "g2p_unstable_host", "g2p_unstable_warnings", "g2p_format_unstable_warning",
    "g2p_unstable_convert_device", "g2p_unstable_convert_host", "g2p_unstable_convert_warnings",
    "g2p_filter_device", "g2p_filter_host",
    "g2p_filter_job_create", "g2p_filter_job_load", "g2p_filter_job_decide", "g2p_filter_job_emit", "g2p_filter_job_get_stats",
    "g2p_filter_job_destroy",
)


class G2PError(RuntimeError):
    pass


class Result(ctypes.Structure):
    """struct g2p_result (include/g2p.h)."""
    _fields_ = [
        ("n_records", ctypes.c_uint64),
        ("out_bytes", ctypes.c_uint64),
        ("rec_status", ctypes.c_uint32),
        ("rec_aux", ctypes.c_uint32),
        ("err_record", ctypes.c_uint64),
        ("err_name_off", ctypes.c_uint64),
        ("err_name_len", ctypes.c_uint32),
        ("gpu_launches", ctypes.c_uint32),
        ("device_ms", ctypes.c_float),
        ("emit_ms", ctypes.c_float),
        ("size_ms", ctypes.c_float),
        ("index_ms", ctypes.c_float),
        ("n_delegated", ctypes.c_uint32),
        ("n_long", ctypes.c_uint32),
        ("fused_ms", ctypes.c_float),
        ("n_fused", ctypes.c_uint32),
        ("unstable_ms", ctypes.c_float),
        ("stage", ctypes.c_uint32),
        ("mid_bytes", ctypes.c_uint64),
        ("par_ms", ctypes.c_float),
        ("n_par", ctypes.c_uint32),
    ]


class FilterParams(ctypes.Structure):
    """struct g2p_filter_params (include/g2p.h): gaffilter's options."""
    _fields_ = [("ratio", ctypes.c_double), ("min_overlap_pct", ctypes.c_double), ("min_identity", ctypes.c_double),
                ("min_overlap_len", ctypes.c_int64), ("min_block_len", ctypes.c_int64), ("min_mapq", ctypes.c_int64),
                ("is_paf", ctypes.c_int32), ("pad", ctypes.c_int32)]


class FilterResult(ctypes.Structure):
    """struct g2p_filter_result (include/g2p.h)."""
    _fields_ = [("n_loaded", ctypes.c_uint64), ("n_filtered", ctypes.c_uint64), ("filtered_len", ctypes.c_uint64), ("out_bytes", ctypes.c_uint64),
                ("rec_status", ctypes.c_uint32), ("gpu_launches", ctypes.c_uint32), ("err_record", ctypes.c_uint64),
                ("device_ms", ctypes.c_float), ("pad", ctypes.c_uint32)]


class FilterJobStats(ctypes.Structure):
    """struct g2p_filter_job_stats (include/g2p.h)."""
    _fields_ = [("load_ms", ctypes.c_double), ("decide_ms", ctypes.c_double), ("emit_ms", ctypes.c_double),
                ("h2d_bytes", ctypes.c_uint64), ("d2h_bytes", ctypes.c_uint64)]


class Warn(ctypes.Structure):
    """struct g2p_warn (include/g2p.h)."""
    _fields_ = [("record", ctypes.c_uint64), ("out_off", ctypes.c_uint64), ("out_len", ctypes.c_uint64)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise G2PError(
            "%s is missing: build it with `make` (nvcc, sm_100a). There is no CPU fallback for this path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, cp, sz = ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t
    lib.g2p_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    lib.g2p_create.restype = ctypes.c_int
    lib.g2p_destroy.argtypes = [vp]
    lib.g2p_destroy.restype = None
    lib.g2p_last_error.argtypes = [vp]
    lib.g2p_last_error.restype = cp
    lib.g2p_host_alloc.argtypes = [sz]
    lib.g2p_host_alloc.restype = vp
    lib.g2p_host_free.argtypes = [vp]
    lib.g2p_host_free.restype = None
    lib.g2p_copy_to_device.argtypes = [vp, vp, sz]
    lib.g2p_copy_to_device.restype = ctypes.c_int
    lib.g2p_copy_to_host.argtypes = [vp, vp, sz]
    lib.g2p_copy_to_host.restype = ctypes.c_int
    lib.g2p_load_lengths.argtypes = [vp, vp, sz]
    lib.g2p_load_lengths.restype = ctypes.c_int
    lib.g2p_table_entries.argtypes = [vp]
    lib.g2p_table_entries.restype = ctypes.c_uint64
    lib.g2p_convert_device.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result), vp]
    lib.g2p_convert_device.restype = ctypes.c_int
    lib.g2p_convert_host.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result)]
    lib.g2p_convert_host.restype = ctypes.c_int
    lib.g2p_index_lines.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_uint64), vp]
    lib.g2p_index_lines.restype = ctypes.c_int
    lib.g2p_format_error.argtypes = [ctypes.POINTER(Result), vp, sz, vp, sz]
    lib.g2p_format_error.restype = ctypes.c_int
    lib.g2p_load_rgfa.argtypes = [vp, vp, sz, ctypes.POINTER(ctypes.c_int), vp, sz]
    lib.g2p_load_rgfa.restype = ctypes.c_int
    lib.g2p_share_rgfa.argtypes = [vp, vp]
    lib.g2p_share_rgfa.restype = ctypes.c_int
    lib.g2p_rgfa_node_lengths.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(sz)]
    lib.g2p_rgfa_node_lengths.restype = ctypes.c_int
    lib.g2p_unstable_device.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result), vp]
    lib.g2p_unstable_device.restype = ctypes.c_int
    lib.g2p_unstable_host.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result)]
    lib.g2p_unstable_host.restype = ctypes.c_int
    lib.g2p_unstable_convert_device.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result), vp]
    lib.g2p_unstable_convert_device.restype = ctypes.c_int
    lib.g2p_unstable_convert_host.argtypes = [vp, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(Result)]
    lib.g2p_unstable_convert_host.restype = ctypes.c_int
    lib.g2p_unstable_convert_warnings.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(sz)]
    lib.g2p_unstable_convert_warnings.restype = ctypes.c_int
    lib.g2p_filter_device.argtypes = [vp, vp, sz, ctypes.POINTER(FilterParams), ctypes.POINTER(vp), ctypes.POINTER(FilterResult), vp]
    lib.g2p_filter_device.restype = ctypes.c_int
    lib.g2p_filter_host.argtypes = [vp, vp, sz, ctypes.POINTER(FilterParams), ctypes.POINTER(vp), ctypes.POINTER(FilterResult)]
    lib.g2p_filter_host.restype = ctypes.c_int
    lib.g2p_filter_job_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.POINTER(FilterParams), ctypes.POINTER(vp)]
    lib.g2p_filter_job_create.restype = ctypes.c_int
    lib.g2p_filter_job_load.argtypes = [vp, ctypes.c_uint64, vp, sz]
    lib.g2p_filter_job_load.restype = ctypes.c_int
    lib.g2p_filter_job_decide.argtypes = [vp, ctypes.POINTER(FilterResult)]
    lib.g2p_filter_job_decide.restype = ctypes.c_int
    lib.g2p_filter_job_emit.argtypes = [vp, ctypes.c_uint64, vp, sz, ctypes.POINTER(vp), ctypes.POINTER(FilterResult)]
    lib.g2p_filter_job_emit.restype = ctypes.c_int
    lib.g2p_filter_job_get_stats.argtypes = [vp, ctypes.POINTER(FilterJobStats)]
    lib.g2p_filter_job_get_stats.restype = ctypes.c_int
    lib.g2p_filter_job_destroy.argtypes = [vp]
    lib.g2p_filter_job_destroy.restype = None
    lib.g2p_unstable_warnings.argtypes = [vp, ctypes.POINTER(ctypes.POINTER(Warn)), ctypes.POINTER(sz)]
    lib.g2p_unstable_warnings.restype = ctypes.c_int
    lib.g2p_format_unstable_warning.argtypes = [vp, vp, sz, vp, sz]
    lib.g2p_format_unstable_warning.restype = ctypes.c_int
    return lib


lib = _load()


def _bytes_at(addr, n):
    """bytes of n bytes at a raw address (ctypes.string_at takes an int-sized length: not enough for > 2 GiB)."""
    return bytes((ctypes.c_char * n).from_address(addr)) if n else b""


def _buf_ptr(b):
    """(address, length, keepalive) of a bytes / bytearray / memoryview / (addr, n) pair."""
    if isinstance(b, tuple):
        return int(b[0]), int(b[1]), None
    if isinstance(b, bytes):
        return ctypes.cast(ctypes.c_char_p(b), ctypes.c_void_p).value or 0, len(b), b
    mv = memoryview(b).cast("B")
    if mv.readonly:
        bb = bytes(mv)
        return ctypes.cast(ctypes.c_char_p(bb), ctypes.c_void_p).value or 0, len(bb), bb
    arr = (ctypes.c_char * len(mv)).from_buffer(mv)
    return ctypes.addressof(arr), len(mv), arr


class Converter:
    """One conversion context bound to one GPU (g2p_ctx)."""

    def __init__(self, device=0):
        h = ctypes.c_void_p()
        rc = lib.g2p_create(int(device), ctypes.byref(h))
        if rc != G2P_OK:
            raise G2PError("g2p_create(device=%d) failed with %d: no usable CUDA device; this library has no CPU path" % (device, rc))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib.g2p_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc):
        if rc != G2P_OK:
            raise G2PError("libg2p error %d: %s" % (rc, lib.g2p_last_error(self._h).decode("latin-1")))

    def load_lengths(self, tsv):
        """get_len_map (reference gaf2paf_main.cpp:22-45).  Returns False where the reference would abort."""
        addr, n, keep = _buf_ptr(tsv)
        rc = lib.g2p_load_lengths(self._h, addr, n)
        if rc == G2P_E_TABLE:
            return False
        self._check(rc)
        return True

    @property
    def table_entries(self):
        return lib.g2p_table_entries(self._h)

    def convert_host(self, gaf):
        """GAF text in host memory -> (paf bytes, Result).  H2D, device pipeline, D2H."""
        addr, n, keep = _buf_ptr(gaf)
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_convert_host(self._h, addr, n, ctypes.byref(out), ctypes.byref(res)))
        return _bytes_at(out.value, res.out_bytes), res

    def convert_host_raw(self, addr, n):
        """Like convert_host for a raw (pinned) host address; returns (out address, Result) without copying."""
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_convert_host(self._h, addr, n, ctypes.byref(out), ctypes.byref(res)))
        return out.value, res

    def convert_device(self, d_ptr, n, stream=0):
        """Device-resident GAF (16-byte aligned device address) -> (device address of PAF, Result)."""
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_convert_device(self._h, d_ptr, n, ctypes.byref(out), ctypes.byref(res), stream or None))
        return out.value, res

    def index_lines(self, d_ptr, n, stream=0):
        """Line index only -> (device address of uint32 starts[n_lines+1], n_lines)."""
        starts = ctypes.c_void_p()
        nl = ctypes.c_uint64()
        self._check(lib.g2p_index_lines(self._h, d_ptr, n, ctypes.byref(starts), ctypes.byref(nl), stream or None))
        return starts.value, nl.value

    # ---- gaf2unstable
    def load_rgfa(self, rgfa):
        """get_unstable_mapping + rgfa2contig (reference gaf2unstable_main.cpp:34-68, rgfa-split.cpp:35-161).
        Returns (ok, reference exit code, reference stderr text)."""
        addr, n, keep = _buf_ptr(rgfa)
        code = ctypes.c_int()
        msg = ctypes.create_string_buffer(1 << 16)
        rc = lib.g2p_load_rgfa(self._h, addr, n, ctypes.byref(code), msg, len(msg))
        if rc == G2P_E_TABLE:
            return False, code.value, msg.value.decode("latin-1")
        self._check(rc)
        return True, 0, ""

    def share_rgfa(self, src):
        """Take the rGFA tables ``src`` (another :class:`Converter`) loaded with :meth:`load_rgfa`, without reading the
        rGFA again (g2p_share_rgfa).  Raises :class:`G2PError` when ``src`` has none."""
        self._check(lib.g2p_share_rgfa(self._h, src._h))

    def node_lengths(self):
        """Contents of the -o file of gaf2unstable."""
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(lib.g2p_rgfa_node_lengths(self._h, ctypes.byref(p), ctypes.byref(n)))
        return ctypes.string_at(p.value, n.value) if n.value else b""

    def unstable_host(self, gaf):
        """Stable-coordinate GAF in host memory -> (node-coordinate GAF bytes, Result, warning texts)."""
        addr, n, keep = _buf_ptr(gaf)
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_unstable_host(self._h, addr, n, ctypes.byref(out), ctypes.byref(res)))
        data = _bytes_at(out.value, res.out_bytes)
        wp, wn = ctypes.POINTER(Warn)(), ctypes.c_size_t()
        self._check(lib.g2p_unstable_warnings(self._h, ctypes.byref(wp), ctypes.byref(wn)))
        warns = []
        for i in range(wn.value):
            w = wp[i]
            line = data[w.out_off:w.out_off + w.out_len]
            buf = ctypes.create_string_buffer(len(line) + 4096)
            lib.g2p_format_unstable_warning(self._h, line, len(line), buf, len(buf))
            warns.append(buf.value.decode("latin-1"))
        return data, res, warns

    def unstable_convert_host(self, gaf):
        """``gaf2unstable gaf -g rgfa -o L | gaf2paf - -l L`` in one call (the intermediate GAF stays on the device):
        -> (paf bytes, Result, stderr text of the gaf2unstable stage)."""
        addr, n, keep = _buf_ptr(gaf)
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_unstable_convert_host(self._h, addr, n, ctypes.byref(out), ctypes.byref(res)))
        return _bytes_at(out.value, res.out_bytes), res, self._convert_warnings()

    def unstable_convert_host_raw(self, addr, n):
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_unstable_convert_host(self._h, addr, n, ctypes.byref(out), ctypes.byref(res)))
        return out.value, res

    def unstable_convert_device(self, d_ptr, n, stream=0):
        out = ctypes.c_void_p()
        res = Result()
        self._check(lib.g2p_unstable_convert_device(self._h, d_ptr, n, ctypes.byref(out), ctypes.byref(res), stream or None))
        return out.value, res

    def _convert_warnings(self):
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        self._check(lib.g2p_unstable_convert_warnings(self._h, ctypes.byref(p), ctypes.byref(n)))
        return ctypes.string_at(p.value, n.value).decode("latin-1") if n.value else ""

    # ---- gaffilter
    @staticmethod
    def filter_params(ratio=0.0, min_overlap=0.0, min_identity=0.0, min_overlap_length=0, min_block_length=0, min_mapq=0, paf=False):
        """gaffilter's options; -r / -m / -i go through std::stof in the reference: the values are rounded to float here too."""
        f32 = lambda x: ctypes.c_float(x).value
        return FilterParams(f32(ratio), f32(min_overlap), f32(min_identity), int(min_overlap_length), int(min_block_length), int(min_mapq), 1 if paf else 0, 0)

    def filter_host(self, text, params):
        """``gaffilter [options] <text>``: -> (kept records as the reference prints them, FilterResult)."""
        addr, n, keep = _buf_ptr(text)
        out = ctypes.c_void_p()
        res = FilterResult()
        self._check(lib.g2p_filter_host(self._h, addr, n, ctypes.byref(params), ctypes.byref(out), ctypes.byref(res)))
        return _bytes_at(out.value, res.out_bytes), res

    def filter_device(self, d_ptr, n, params, stream=0):
        """Filter text that is already on the device (e.g. the PAF g2p_convert_device just made): -> (device address, FilterResult)."""
        out = ctypes.c_void_p()
        res = FilterResult()
        self._check(lib.g2p_filter_device(self._h, d_ptr, n, ctypes.byref(params), ctypes.byref(out), ctypes.byref(res), stream or None))
        return out.value, res

    @staticmethod
    def format_error(res, gaf):
        addr, n, keep = _buf_ptr(gaf)
        buf = ctypes.create_string_buffer(2048)
        lib.g2p_format_error(ctypes.byref(res), addr, n, buf, len(buf))
        return buf.value.decode("latin-1")


class FilterJob:
    """gaffilter on inputs of any size over one or more :class:`Converter` contexts (g2p_filter_job_*): ``load`` every
    newline-aligned chunk (numbered from 0 in input order; chunk c runs on converters[c % len(converters)]), ``decide``
    once (-> the FilterResult of the whole input), then ``emit`` every chunk again (-> its kept records)."""

    def __init__(self, converters, params):
        self._cvs = list(converters)
        hs = (ctypes.c_void_p * len(self._cvs))(*[cv._h.value for cv in self._cvs])
        h = ctypes.c_void_p()
        self._params = params
        rc = lib.g2p_filter_job_create(hs, len(self._cvs), ctypes.byref(params), ctypes.byref(h))
        if rc != G2P_OK:
            raise G2PError("g2p_filter_job_create failed with %d" % rc)
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib.g2p_filter_job_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc, chunk=0):
        if rc != G2P_OK:
            self._cvs[chunk % len(self._cvs)]._check(rc)

    def load(self, chunk, text):
        addr, n, keep = _buf_ptr(text)
        self._check(lib.g2p_filter_job_load(self._h, chunk, addr, n), chunk)

    def decide(self):
        res = FilterResult()
        self._check(lib.g2p_filter_job_decide(self._h, ctypes.byref(res)))
        return res

    def emit(self, chunk, text):
        """-> (kept records of the chunk, FilterResult of the chunk)."""
        addr, n, keep = _buf_ptr(text)
        out = ctypes.c_void_p()
        res = FilterResult()
        self._check(lib.g2p_filter_job_emit(self._h, chunk, addr, n, ctypes.byref(out), ctypes.byref(res)), chunk)
        return _bytes_at(out.value, res.out_bytes), res

    def stats(self):
        s = FilterJobStats()
        lib.g2p_filter_job_get_stats(self._h, ctypes.byref(s))
        return s


def copy_to_host(d_ptr, n):
    """Device address -> bytes (cudaMemcpy through the C-ABI)."""
    buf = ctypes.create_string_buffer(max(1, n))
    if n and lib.g2p_copy_to_host(buf, d_ptr, n) != G2P_OK:
        raise G2PError("g2p_copy_to_host failed")
    return buf.raw[:n]


def copy_to_device(d_ptr, data):
    addr, n, keep = _buf_ptr(data)
    if n and lib.g2p_copy_to_device(d_ptr, addr, n) != G2P_OK:
        raise G2PError("g2p_copy_to_device failed")


def exit_code(res):
    """Process exit status of the reference for this result (0, 1 or 134)."""
    if res.rec_status == REC_OK:
        return 0
    return 134 if res.rec_status >= REC_ABORT else 1


def gaf2paf(gaf, lengths, device=0, converter=None):
    """``gaf2paf -l <lengths> <gaf>``: returns (stdout bytes, exit code, stderr text)."""
    cv = converter or Converter(device)
    try:
        if not cv.load_lengths(lengths):
            return b"", 134, "terminate called after throwing an instance of 'std::invalid_argument'\n  what():  stol\n"
        out, res = cv.convert_host(gaf)
        rc = exit_code(res)
        err = Converter.format_error(res, gaf) if rc else ""
        return out, rc, err
    finally:
        if converter is None:
            cv.close()


def shard_ranges(buf, n_shards):
    """Newline-aligned byte ranges [(a, b), ...] covering ``buf`` (multi-GPU sharding, SURVEY.md §8e):
    cut the byte range into n contiguous pieces and move every cut forward to just after the next newline."""
    n = len(buf)
    cuts = [0]
    for i in range(1, n_shards):
        p = max(cuts[-1], n * i // n_shards)
        if p > 0 and p < n and buf[p - 1:p] != b"\n":
            q = buf.find(b"\n", p)
            p = n if q < 0 else q + 1
        cuts.append(min(p, n))
    cuts.append(n)
    return [(cuts[i], cuts[i + 1]) for i in range(n_shards)]
