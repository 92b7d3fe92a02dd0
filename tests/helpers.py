"""Shared test plumbing: loads the two CPU checkers (oracle port, compiled reference) with ctypes
and builds the input zoo modelled on the reference fuzzers' buffers
(programs/fuzzer.c:157-161: noise, P=1%, 15%, 90%, constant)."""
import ctypes as C
import hashlib
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
PORT_SO = os.path.join(ORACLE_DIR, "_build", "libfse_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libfse_ref.so")

sz = C.c_size_t
vp = C.c_void_p
u = C.c_uint
ERR_MAX = 9


def is_error(r):
    return r > (2 ** 64 - ERR_MAX)


def err_code(r):
    return (2 ** 64 - r) if is_error(r) else 0


def _sig(fn, res, *args):
    fn.restype = res
    fn.argtypes = list(args)
    return fn


_port = None


def load_port():
    """our plain-C restatement (always buildable: gcc only)"""
    global _port
    if _port is None:
        src = os.path.join(ORACLE_DIR, "fse_oracle.c")
        if (not os.path.exists(PORT_SO)) or os.path.getmtime(PORT_SO) < os.path.getmtime(src):
            subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "port"])
        L = C.CDLL(PORT_SO)
        P = C.POINTER
        _sig(L.orc_hist_count, sz, P(u), P(u), vp, sz)
        _sig(L.orc_optimal_tablelog, u, u, sz, u, u)
        _sig(L.orc_fse_normalize, sz, P(C.c_short), u, P(u), sz, u)
        _sig(L.orc_fse_ncount_bound, sz, u, u)
        _sig(L.orc_fse_write_ncount, sz, vp, sz, P(C.c_short), u, u)
        _sig(L.orc_fse_read_ncount, sz, P(C.c_short), P(u), P(u), vp, sz)
        _sig(L.orc_fse_build_ctable, sz, vp, P(C.c_short), u, u)
        _sig(L.orc_fse_build_dtable, sz, vp, P(C.c_short), u, u)
        _sig(L.orc_fse_build_dtable_u16, sz, vp, P(C.c_short), u, u)
        _sig(L.orc_fse_encode, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_fse_decode, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_fse_compress2, sz, vp, sz, vp, sz, u, u)
        _sig(L.orc_fse_decompress, sz, vp, sz, vp, sz)
        _sig(L.orc_fse_compress_u16, sz, vp, sz, vp, sz, u, u)
        _sig(L.orc_fse_decompress_u16, sz, vp, sz, vp, sz)
        _sig(L.orc_huf_build_ctable, sz, vp, P(u), u, u)
        _sig(L.orc_huf_write_ctable, sz, vp, sz, vp, u, u)
        _sig(L.orc_huf_encode4x, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_huf_encode1x, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_huf_compress2, sz, vp, sz, vp, sz, u, u)
        _sig(L.orc_huf_read_stats, sz, vp, sz, vp, P(C.c_uint32), P(C.c_uint32), vp, sz)
        _sig(L.orc_huf_read_dtable_x1, sz, vp, vp, sz)
        _sig(L.orc_huf_read_dtable_x2, sz, vp, vp, sz)
        _sig(L.orc_huf_decode4x2, sz, vp, sz, vp, sz, vp); _sig(L.orc_huf_decode1x2, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_huf_decode4x1, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_huf_decode1x1, sz, vp, sz, vp, sz, vp)
        _sig(L.orc_huf_decompress, sz, vp, sz, vp, sz)
        _sig(L.orc_huf_decompress4x1, sz, vp, sz, vp, sz); _sig(L.orc_huf_decompress4x2, sz, vp, sz, vp, sz)
        _sig(L.orc_huf_select_decoder, u, sz, sz)
        _sig(L.orc_probagen, None, vp, sz, C.c_double)
        _sig(L.orc_gen_u16, None, vp, sz, u, C.c_double, C.c_uint32)
        _sig(L.orc_xxh64, C.c_uint64, vp, sz, C.c_uint64)
        _sig(L.orc_xxh32, C.c_uint32, vp, sz, C.c_uint32)
        _sig(L.orc_compress_blocks, sz, C.c_int, vp, sz, sz, vp, sz, vp, u, u)
        _sig(L.orc_decompress_blocks, sz, C.c_int, vp, vp, sz, sz, vp, sz, vp, vp)
        _port = L
    return _port


_ref = None


def load_ref():
    """the unmodified reference library.  Inside a test: as recorded for that test (reference_calls.py), replayed from
    tests/golden/reference_calls.npz, or the compiled library itself while recording.  Elsewhere (tests/golden/make_golden.py,
    smoke()): the library compiled by oracle/Makefile into oracle/_ref, or None where it was not built."""
    global _ref
    import reference_calls
    if reference_calls.active():
        L = reference_calls.current()
    elif _ref is not None:
        return _ref
    elif not os.path.exists(REF_SO):
        return None
    else:
        L = _ref = C.CDLL(REF_SO)
    P = C.POINTER
    _sig(L.HIST_count, sz, P(u), P(u), vp, sz)
    _sig(L.FSE_optimalTableLog, u, u, sz, u)
    _sig(L.HUF_optimalTableLog, u, u, sz, u)
    _sig(L.FSE_normalizeCount, sz, P(C.c_short), u, P(u), sz, u)
    _sig(L.FSE_NCountWriteBound, sz, u, u)
    _sig(L.FSE_writeNCount, sz, vp, sz, P(C.c_short), u, u)
    _sig(L.FSE_readNCount, sz, P(C.c_short), P(u), P(u), vp, sz)
    _sig(L.FSE_buildCTable, sz, vp, P(C.c_short), u, u)
    _sig(L.FSE_buildCTableU16, sz, vp, P(C.c_short), u, u)
    _sig(L.FSE_buildDTable, sz, vp, P(C.c_short), u, u)
    _sig(L.FSE_buildDTableU16, sz, vp, P(C.c_short), u, u)
    _sig(L.FSE_compress_usingCTable, sz, vp, sz, vp, sz, vp)
    _sig(L.FSE_decompress_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.FSE_compress2, sz, vp, sz, vp, sz, u, u)
    _sig(L.FSE_compress, sz, vp, sz, vp, sz)
    _sig(L.FSE_decompress, sz, vp, sz, vp, sz)
    _sig(L.FSE_compressBound, sz, sz)
    _sig(L.FSE_compressU16, sz, vp, sz, vp, sz, u, u)
    _sig(L.FSE_decompressU16, sz, vp, sz, vp, sz)
    _sig(L.HUF_buildCTable, sz, vp, P(u), u, u)
    _sig(L.HUF_writeCTable, sz, vp, sz, vp, u, u)
    _sig(L.HUF_compress4X_usingCTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_compress1X_usingCTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_compress2, sz, vp, sz, vp, sz, u, u)
    _sig(L.HUF_compress, sz, vp, sz, vp, sz)
    _sig(L.HUF_readStats, sz, vp, sz, vp, P(C.c_uint32), P(C.c_uint32), vp, sz)
    _sig(L.HUF_readDTableX1, sz, vp, vp, sz)
    _sig(L.HUF_readDTableX2, sz, vp, vp, sz)
    _sig(L.HUF_decompress4X2_usingDTable, sz, vp, sz, vp, sz, vp); _sig(L.HUF_decompress1X2_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_readDTableX2, sz, vp, vp, sz)
    _sig(L.HUF_decompress4X2_usingDTable, sz, vp, sz, vp, sz, vp); _sig(L.HUF_decompress1X2_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_decompress4X1_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_decompress4X2_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_decompress4X_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_decompress1X1_usingDTable, sz, vp, sz, vp, sz, vp)
    _sig(L.HUF_decompress, sz, vp, sz, vp, sz)
    _sig(L.HUF_decompress4X1, sz, vp, sz, vp, sz)
    _sig(L.HUF_decompress4X2, sz, vp, sz, vp, sz)
    _sig(L.HUF_selectDecoder, C.c_uint32, sz, sz)
    _sig(L.refshim_compress_blocks, C.c_double, C.c_int, vp, sz, sz, vp, sz, vp, u, u, C.c_int)
    _sig(L.refshim_decompress_blocks, C.c_double, C.c_int, vp, vp, sz, sz, vp, sz, vp, vp, C.c_int)
    return L


def ptr(a):
    """raw pointer of a numpy array / bytearray as c_void_p"""
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(vp)
    return C.cast((C.c_char * len(a)).from_buffer(a), vp)


def probagen(n, p):
    out = np.empty(n, dtype=np.uint8)
    load_port().orc_probagen(ptr(out), n, float(p))
    return out


def gen_u16(n, start=240, p=0.5, seed=1):
    out = np.empty(n, dtype=np.uint16)
    load_port().orc_gen_u16(ptr(out), n, start, float(p), seed)
    return out


def zoo(rng, n):
    """one random buffer of length n from the fuzzers' buffer zoo (+ a few nastier shapes)"""
    kind = int(rng.integers(0, 9))
    if kind == 0:
        return rng.integers(0, 256, n, dtype=np.uint8)                      # noise
    if kind == 1:
        return np.full(n, int(rng.integers(0, 256)), dtype=np.uint8)        # constant (RLE)
    if kind in (2, 3, 4):
        p = [0.01, 0.15, 0.90][kind - 2]
        off = int(rng.integers(0, 1 << 16))
        return probagen(off + n, p)[off:]
    if kind == 5:                                                          # geometric over a random alphabet
        k = int(rng.integers(2, 257))
        q = float(rng.uniform(0.02, 0.6))
        v = np.minimum(rng.geometric(q, n) - 1, k - 1).astype(np.uint8)
        perm = rng.permutation(256).astype(np.uint8)
        return perm[v]
    if kind == 6:                                                          # few symbols, one dominant
        v = (rng.random(n) < float(rng.uniform(0.001, 0.2))).astype(np.uint8) * rng.integers(1, 256, n, dtype=np.uint8)
        return v
    if kind == 7:                                                          # zipf-like, wide alphabet (deep Huffman trees)
        w = 1.0 / np.arange(1, 257) ** float(rng.uniform(0.8, 2.5))
        return rng.choice(256, n, p=w / w.sum()).astype(np.uint8)
    v = rng.integers(0, int(rng.integers(2, 40)), n, dtype=np.uint8)      # small flat alphabet
    return v


def small_vectors():
    """the inputs of tests/golden/vectors_small.npz in order, as (codec, bytes): 0 FSE and 1 Huff0 on the same
    ragged / edge-sized byte buffer from the zoo, then 2 FSE-U16 on 16-bit symbols"""
    rng = np.random.default_rng(20260922)
    sizes = [0, 1, 2, 3, 4, 7, 11, 12, 13, 15, 16, 17, 31, 64, 100, 255, 256, 1000, 1001, 1499, 1500, 4096, 8191, 32765, 32766, 32767, 32768, 65536, 131072]
    for n in sizes + [int(rng.integers(20, 40000)) for _ in range(40)]:
        d = np.ascontiguousarray(zoo(rng, n))
        yield 0, d
        yield 1, d
    for n in (2, 3, 16, 1000, 16384, 16383, 40000):
        yield 2, np.ascontiguousarray(gen_u16(n + 50, 240, float(rng.uniform(0.05, 0.8)), int(rng.integers(1, 1 << 30)))[50:]).view(np.uint8)


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def rand_size(rng, hi=128 * 1024):
    r = rng.random()
    if r < 0.25:
        return int(rng.integers(0, 64))
    if r < 0.5:
        return int(rng.integers(64, 4096))
    return int(rng.integers(4096, hi + 1))
