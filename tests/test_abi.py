"""CPU-side checks of the C-ABI boundary: libfse_b200.so builds (nvcc cross-compiles without a GPU),
loads, and exports every symbol include/fse_b200.h declares.  No compute calls here."""
import ctypes
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "fse_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:FSEB200|FSE|HUF|HIST)_\w+)\s*\(", text)))


def test_header_declares_the_north_star_surface():
    names = _declared()
    for must in ("FSE_compress", "FSE_decompress", "HUF_compress", "HUF_decompress", "FSE_buildCTable", "FSE_buildDTable",
                 "HIST_count", "FSE_compress2", "HUF_compress2", "FSE_compressU16", "FSE_decompressU16",
                 "FSEB200_HUF_decompress_batch", "FSEB200_HUF_compress_batch", "FSEB200_FSE_compress_batch",
                 "FSEB200_FSE_decompress_batch"):
        assert must in names


def test_library_builds_loads_and_exports_everything():
    import finitestateentropy_b200 as fb
    from finitestateentropy_b200 import _build
    path = _build.build_lib()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    missing = [n for n in _declared() if not hasattr(lib, n)]
    assert not missing, missing
    exported = subprocess.check_output(["nm", "-D", "--defined-only", path]).decode()
    assert " T HUF_decompress" in exported and " T FSEB200_HUF_decompress_batch" in exported
    # scalar helpers are host arithmetic and may be called without a GPU
    lib.FSE_compressBound.restype = ctypes.c_size_t; lib.FSE_compressBound.argtypes = [ctypes.c_size_t]
    assert lib.FSE_compressBound(32768) == 33548                      # SURVEY.md section 8, programs/bench.c:355
    lib.FSE_isError.argtypes = [ctypes.c_size_t]
    assert lib.FSE_isError(2 ** 64 - 4) == 1 and lib.FSE_isError(33548) == 0
    lib.FSE_getErrorName.restype = ctypes.c_char_p; lib.FSE_getErrorName.argtypes = [ctypes.c_size_t]
    assert lib.FSE_getErrorName(2 ** 64 - 4) == b"Corrupted block detected"
    assert lib.FSE_versionNumber() == 900
    lib.FSE_optimalTableLog.argtypes = [ctypes.c_uint, ctypes.c_size_t, ctypes.c_uint]
    assert lib.FSE_optimalTableLog(12, 32768, 52) == 12 and lib.FSE_optimalTableLog(12, 16384, 286) == 11
    assert fb.compress_bound(32768) == 33548


def test_product_does_not_touch_the_oracle():
    """the product tree must not reference oracle/ (judge rule: oracle is test infrastructure only)"""
    bad = []
    for base in ("finitestateentropy_b200", "include"):
        for dp, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c")):
                    t = open(os.path.join(dp, f), errors="ignore").read()
                    if re.search(r"fse_oracle|libfse_ref|oracle/_ref|orc_", t) and f != "_build.py":
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_constant_pattern_tables_match_the_reference():
    """FSE_buildCTable_raw/_rle and FSE_buildDTable_raw/_rle are host-side fills of the ABI layouts: word-equal with the
    compiled reference (fse_compress.c:498-551, fse_decompress.c:134-176)"""
    import numpy as np
    from helpers import load_ref, ptr
    from finitestateentropy_b200 import _build
    ref = load_ref()
    lib = ctypes.CDLL(_build.build_lib())
    for L in (lib, ref):
        for n in ("FSE_buildCTable_raw", "FSE_buildDTable_raw"):
            f = getattr(L, n); f.restype = ctypes.c_size_t; f.argtypes = [ctypes.c_void_p, ctypes.c_uint]
        for n in ("FSE_buildCTable_rle", "FSE_buildDTable_rle"):
            f = getattr(L, n); f.restype = ctypes.c_size_t; f.argtypes = [ctypes.c_void_p, ctypes.c_ubyte]
    for nb in range(0, 9):
        a = np.zeros(1 + 128 + 2 * 256 + 8, np.uint32); b = np.zeros_like(a)
        ra, rb = lib.FSE_buildCTable_raw(ptr(a), nb), ref.FSE_buildCTable_raw(ptr(b), nb)
        assert ra == rb and np.array_equal(a, b)
        a = np.zeros(1 + 256 + 8, np.uint32); b = np.zeros_like(a)
        ra, rb = lib.FSE_buildDTable_raw(ptr(a), nb), ref.FSE_buildDTable_raw(ptr(b), nb)
        assert ra == rb and np.array_equal(a, b)
    for sym in (0, 1, 77, 255):
        a = np.zeros(2 + 2 * 256 + 8, np.uint32); b = np.zeros_like(a)
        assert lib.FSE_buildCTable_rle(ptr(a), sym) == ref.FSE_buildCTable_rle(ptr(b), sym) == 0 and np.array_equal(a, b)
        a = np.zeros(4, np.uint32); b = np.zeros_like(a)
        assert lib.FSE_buildDTable_rle(ptr(a), sym) == ref.FSE_buildDTable_rle(ptr(b), sym) == 0 and np.array_equal(a, b)


def test_prototypes_have_the_reference_arity():
    """Every reference-named entry point declared in include/fse_b200.h takes as many parameters as the declaration of the
    same name in the reference's own headers (lib/fse.h, huf.h, hist.h, fseU16.h), as recorded from them (reference_calls.py;
    recording reads the headers under $FSE_REFERENCE_DIR/lib)."""
    import json
    from helpers import load_ref

    def protos(text):
        text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S); text = re.sub(r"//[^\n]*", " ", text)
        out = {}
        for m in re.finditer(r"\b((?:FSE|HUF|HIST)_\w+)\s*\(([^;{}()]*)\)\s*;", text):
            args = m.group(2).strip()
            out[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
        return out
    def read_theirs():
        theirs = {}
        for h in ("fse.h", "huf.h", "hist.h", "fseU16.h"):
            theirs.update(protos(open(os.path.join(os.environ["FSE_REFERENCE_DIR"], "lib", h)).read()))
        return json.dumps(theirs, sort_keys=True)
    theirs = json.loads(load_ref().value("prototype arity", read_theirs))
    ours = protos(open(os.path.join(ROOT, "include", "fse_b200.h")).read())
    common = sorted(set(ours) & set(theirs))
    assert len(common) >= 40, common
    bad = [(n, ours[n], theirs[n]) for n in common if ours[n] != theirs[n]]
    assert not bad, bad


def test_ctable_helpers_match_the_reference():
    """HUF_getNbBits / HUF_estimateCompressedSize / HUF_validateCTable: host arithmetic on CTable cells, equal to the reference"""
    import numpy as np
    from helpers import load_ref, ptr
    from finitestateentropy_b200 import _build
    ref = load_ref()
    lib = ctypes.CDLL(_build.build_lib())
    U = ctypes.c_uint
    for L in (lib, ref):
        L.HUF_getNbBits.restype = U; L.HUF_getNbBits.argtypes = [ctypes.c_void_p, U]
        L.HUF_estimateCompressedSize.restype = ctypes.c_size_t; L.HUF_estimateCompressedSize.argtypes = [ctypes.c_void_p, ctypes.c_void_p, U]
        L.HUF_validateCTable.restype = ctypes.c_int; L.HUF_validateCTable.argtypes = [ctypes.c_void_p, ctypes.c_void_p, U]
    ref.HUF_buildCTable.restype = ctypes.c_size_t; ref.HUF_buildCTable.argtypes = [ctypes.c_void_p, ctypes.c_void_p, U, U]
    rng = np.random.default_rng(5)
    for it in range(20):
        msv = int(rng.integers(1, 256))
        cnt = rng.integers(0, 500, 256).astype(np.uint32); cnt[msv] = max(1, int(cnt[msv])); cnt[0] = max(1, int(cnt[0]))
        ct = np.zeros(256, np.uint32)
        r = ref.HUF_buildCTable(ptr(ct), ptr(cnt), msv, 11)
        assert r < 2 ** 63
        assert lib.HUF_estimateCompressedSize(ptr(ct), ptr(cnt), msv) == ref.HUF_estimateCompressedSize(ptr(ct), ptr(cnt), msv)
        assert lib.HUF_validateCTable(ptr(ct), ptr(cnt), msv) == ref.HUF_validateCTable(ptr(ct), ptr(cnt), msv) == 1
        cnt2 = cnt.copy(); z = [s for s in range(msv + 1) if (ct[s] >> 16) & 0xFF == 0]
        if z:
            cnt2[z[0]] = 3
            assert lib.HUF_validateCTable(ptr(ct), ptr(cnt2), msv) == ref.HUF_validateCTable(ptr(ct), ptr(cnt2), msv) == 0
        for s in (0, msv // 2, msv):
            assert lib.HUF_getNbBits(ptr(ct), s) == ref.HUF_getNbBits(ptr(ct), s)
