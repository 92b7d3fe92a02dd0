"""Parity of every CUDA codec path against the CPU checker through the C-ABI (-m gpu):
identical compressed bytes and return values (incl. the in-band 0 / 1), both cross-decodes,
golden vectors, table images, and the size-independent round-trip property at larger sizes."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from helpers import ptr, zoo, rand_size, probagen, gen_u16, is_error, small_vectors, sha256
from gpu_common import cpu_compress, cpu_decompress, checker, BLOCK, SLOT
import finitestateentropy_b200 as fb

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
U = C.c_uint


def _dev(a):
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a.view(np.uint8)).cuda()


ENC = {"huf": fb.huf_compress_batch, "fse": fb.fse_compress_batch, "u16": fb.fseu16_compress_batch}
DEC = {"huf": fb.huf_decompress_batch, "fse": fb.fse_decompress_batch, "u16": fb.fseu16_decompress_batch}


def _roundtrip_vs_checker(codec, data, block, msv=255, tl=12, slot=None):
    data = np.ascontiguousarray(data).view(np.uint8)
    slot = slot or (32768 if codec == "u16" and block == 32768 else 512 + block + (block >> 7) + 12)
    want_c, want_cs, _ = cpu_compress(codec, data, block=block, slot=slot, msv=msv, tl=tl)
    d_src = _dev(data)
    cbuf, cs = ENC[codec](d_src, block, slot, msv, tl)
    torch.cuda.synchronize()
    got_cs = cs.cpu().numpy().view(np.uint64)
    got_c = cbuf.cpu().numpy()
    nb = len(want_cs)
    for b in range(nb):
        assert got_cs[b] == want_cs[b], (codec, block, b, int(got_cs[b]), int(want_cs[b]))
        if not is_error(int(want_cs[b])) and want_cs[b] > 1:
            a = got_c[b * slot: b * slot + int(want_cs[b])]; w = want_c[b * slot: b * slot + int(want_cs[b])]
            assert np.array_equal(a, w), (codec, block, b, int(np.nonzero(a != w)[0][0]))
        if codec == "huf" and want_cs[b] == 1:
            assert got_c[b * slot] == want_c[b * slot]
    # GPU decode of GPU output, CPU decode of GPU output
    want_out, want_res = cpu_decompress(codec, got_c, got_cs.copy(), data, block=block, slot=slot)
    out, res = DEC[codec](cbuf, cs, len(data), block, slot, orig=d_src)
    torch.cuda.synchronize()
    res = res.cpu().numpy().view(np.uint64); out = out.cpu().numpy()
    for b in range(nb):
        if is_error(int(got_cs[b])):
            continue
        assert res[b] == want_res[b], (codec, block, b, int(res[b]), int(want_res[b]), int(got_cs[b]))
        n = min(block, len(data) - b * block)
        if not is_error(int(want_res[b])):
            assert np.array_equal(out[b * block: b * block + n], data[b * block: b * block + n]), (codec, b)
    return got_cs


@pytest.mark.parametrize("codec,p", [("huf", 0.14), ("huf", 0.80), ("huf", 0.02), ("fse", 0.20), ("fse", 0.80), ("fse", 0.02), ("fse", 0.14)])
def test_probagen_1mib_matches_kat(codec, p):
    """config[0]-style run: 1,048,575 B, 32 blocks, (255,12) -- totals must match SURVEY.md 6.3 / kat_bench.json"""
    data = probagen(1048575, p)
    cs = _roundtrip_vs_checker(codec, data, BLOCK, slot=SLOT)
    kat = {(r["name"], r["codec"]): r for r in json.load(open(os.path.join(HERE, "golden", "kat_bench.json")))}
    rec = kat[("proba%02d" % round(p * 100), codec)]
    assert [int(x) for x in cs] == rec["cSizes"]


def test_u16_matches_kat():
    data = gen_u16(524288, 240, 0.50, 1)
    cs = _roundtrip_vs_checker("u16", data, 32768, msv=0, tl=12, slot=32768)
    rec = [r for r in json.load(open(os.path.join(HERE, "golden", "kat_bench.json"))) if r["codec"] == "u16"][0]
    assert [int(x) for x in cs] == rec["cSizes"]


@pytest.mark.parametrize("codec", ["huf", "fse"])
def test_zoo_blocks(codec):
    rng = np.random.default_rng(21 if codec == "huf" else 22)
    for block in (32768, 4099, 1000, 65536, 131072, 12, 77, 13):
        parts = [zoo(rng, block) for _ in range(int(rng.integers(3, 40)))]
        parts.append(zoo(rng, int(rng.integers(1, block + 1))))
        _roundtrip_vs_checker(codec, np.concatenate(parts), block)


def test_u16_zoo():
    rng = np.random.default_rng(23)
    for block_syms in (16384, 1000, 4099, 3, 2):
        parts = []
        for _ in range(12):
            k = int(rng.integers(0, 3))
            if k == 0:
                parts.append(gen_u16(block_syms, 240, float(rng.uniform(0.05, 0.9)), int(rng.integers(1, 1 << 30))))
            elif k == 1:
                parts.append(rng.integers(0, int(rng.integers(1, 287)), block_syms).astype(np.uint16))
            else:
                parts.append(np.full(block_syms, int(rng.integers(0, 287)), np.uint16))
        data = np.concatenate(parts)
        _roundtrip_vs_checker("u16", data, 2 * block_syms, msv=0, tl=12, slot=2 * block_syms + 600)


def test_golden_small_vectors_through_host_api():
    """tests/golden/vectors_small.npz (inputs regenerated, checked by digest) through the reference-named one-block entry points
    (host pointers)"""
    L = fb.lib()
    for name, res, args in (("FSE_compress2", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, U, U]),
                            ("HUF_compress2", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, U, U]),
                            ("FSE_compressU16", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, U, U]),
                            ("FSE_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
                            ("HUF_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
                            ("FSE_decompressU16", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t])):
        f = getattr(L, name); f.restype = res; f.argtypes = args
    z = np.load(os.path.join(HERE, "golden", "vectors_small.npz"))
    vecs = list(small_vectors())
    assert len(vecs) == int(z["count"][0])
    for k, (codec, d) in enumerate(vecs):
        assert codec == int(z["codec"][k]) and sha256(d) == z["in_sha256"][k], k      # the recorded input
        want = int(z["ret"][k])
        n = len(d)
        if codec == 2:
            dst = np.zeros(n + 600, np.uint8)
            r = L.FSE_compressU16(ptr(dst), n + 592, ptr(d), n // 2, 0, 12)
        else:
            cap = 512 + n + (n >> 7) + 12
            dst = np.zeros(cap + 8, np.uint8)
            r = (L.FSE_compress2 if codec == 0 else L.HUF_compress2)(ptr(dst), cap, ptr(d), n, 255, 12)
        assert r == want, (k, codec, n, r, want)
        if not is_error(r) and r > 1:
            assert sha256(dst[:r]) == z["out_sha256"][k], (k, codec, n)
            out = np.zeros(n + 2, np.uint8)
            if codec == 2:
                assert L.FSE_decompressU16(ptr(out), n // 2, ptr(dst), r) == n // 2
                assert np.array_equal(out[:n], d)
            else:
                dr = (L.FSE_decompress if codec == 0 else L.HUF_decompress)(ptr(out), n, ptr(dst), r)
                if not is_error(dr):
                    assert dr == n and np.array_equal(out[:n], d)


def test_fse_error_verdicts():
    """truncated / corrupted FSE blocks: same verdict and bytes as the CPU decoder (programs/fuzzer.c:253-262)"""
    lib, isref = checker()
    dec = lib.FSE_decompress if isref else lib.orc_fse_decompress
    rng = np.random.default_rng(24)
    block = 4096
    data = np.concatenate([zoo(rng, block) for _ in range(120)])
    cbuf, cs, slot = cpu_compress("fse", data, block=block)
    nb = len(cs); want = np.zeros(nb, np.uint64); wout = np.zeros(len(data), np.uint8)
    for b in range(nb):
        if cs[b] < 2:
            want[b] = block; wout[b * block:(b + 1) * block] = data[b * block:(b + 1) * block]
            continue
        c = cbuf[b * slot: b * slot + int(cs[b])]
        mode = int(rng.integers(0, 3))
        if mode == 0:
            cs[b] = int(rng.integers(2, int(cs[b])))
        elif mode == 1:
            for _ in range(int(rng.integers(1, 4))):
                c[int(rng.integers(0, len(c)))] ^= int(rng.integers(1, 256))
        tmp = np.concatenate([cbuf[b * slot: b * slot + int(cs[b])], np.zeros(32, np.uint8)])
        o = np.zeros(block + 8, np.uint8)
        want[b] = dec(ptr(o), block, ptr(tmp), int(cs[b]))
        wout[b * block:(b + 1) * block] = o[:block]
    guard = torch.full((len(data) + 4096,), 0x5A, dtype=torch.uint8, device="cuda")
    out, res = fb.fse_decompress_batch(_dev(cbuf), _dev(cs), len(data), block, slot, out=guard, orig=_dev(data))
    torch.cuda.synchronize()
    res = res.cpu().numpy().view(np.uint64); out = out.cpu().numpy()
    bad = [(b, int(res[b]), int(want[b])) for b in range(nb) if res[b] != want[b]]
    assert not bad, bad[:10]
    for b in range(nb):
        if not is_error(int(want[b])):
            k = int(want[b])
            assert np.array_equal(out[b * block: b * block + k], wout[b * block: b * block + k]), b
    assert (guard[len(data):] == 0x5A).all()
    assert sum(is_error(int(x)) for x in want) > 5


def test_table_level_api_images():
    """HIST_count / FSE_normalizeCount / NCount / FSE_buildCTable / FSE_buildDTable / HUF_buildCTable /
    HUF_writeCTable / HUF_readStats / HUF_readDTableX1 computed on the GPU vs the CPU checker's images"""
    lib, isref = checker()
    L = fb.lib()
    P = C.POINTER
    def sig(n, *a):
        f = getattr(L, n); f.restype = C.c_size_t; f.argtypes = list(a); return f
    g_hist = sig("HIST_count", P(U), P(U), C.c_void_p, C.c_size_t)
    g_norm = sig("FSE_normalizeCount", P(C.c_short), U, P(U), C.c_size_t, U)
    g_wn = sig("FSE_writeNCount", C.c_void_p, C.c_size_t, P(C.c_short), U, U)
    g_rn = sig("FSE_readNCount", P(C.c_short), P(U), P(U), C.c_void_p, C.c_size_t)
    g_ct = sig("FSE_buildCTable", C.c_void_p, P(C.c_short), U, U)
    g_dt = sig("FSE_buildDTable", C.c_void_p, P(C.c_short), U, U)
    g_hct = sig("HUF_buildCTable", C.c_void_p, P(U), U, U)
    g_hw = sig("HUF_writeCTable", C.c_void_p, C.c_size_t, C.c_void_p, U, U)
    g_hrs = sig("HUF_readStats", C.c_void_p, C.c_size_t, P(C.c_uint32), P(C.c_uint32), P(C.c_uint32), C.c_void_p, C.c_size_t)
    g_hdt = sig("HUF_readDTableX1", C.c_void_p, C.c_void_p, C.c_size_t)
    L.FSE_optimalTableLog.argtypes = [U, C.c_size_t, U]; L.HUF_optimalTableLog.argtypes = [U, C.c_size_t, U]
    rng = np.random.default_rng(25)
    for it in range(25):
        n = int(rng.integers(300, 40000)); d = zoo(rng, n)
        ca = (U * 256)(); cb = (U * 256)(); ma, mb = U(255), U(255)
        ra = g_hist(ca, C.byref(ma), ptr(d), n); rb = lib.HIST_count(cb, C.byref(mb), ptr(d), n)
        assert ra == rb and ma.value == mb.value and list(ca) == list(cb)
        msv = ma.value
        if ra == n or msv == 0:
            continue
        tl = lib.FSE_optimalTableLog(12, n, msv)
        assert tl == L.FSE_optimalTableLog(12, n, msv)
        na = (C.c_short * 256)(); nb_ = (C.c_short * 256)()
        assert g_norm(na, tl, ca, n, msv) == lib.FSE_normalizeCount(nb_, tl, cb, n, msv)
        assert list(na)[:msv + 1] == list(nb_)[:msv + 1]
        ha = np.zeros(600, np.uint8); hb = np.zeros(600, np.uint8)
        wa = g_wn(ptr(ha), 600, na, msv, tl); wb = lib.FSE_writeNCount(ptr(hb), 600, nb_, msv, tl)
        assert wa == wb and bytes(ha[:wa]) == bytes(hb[:wb])
        xa = (C.c_short * 256)(); xb = (C.c_short * 256)(); m1, m2, t1, t2 = U(255), U(255), U(0), U(0)
        assert g_rn(xa, C.byref(m1), C.byref(t1), ptr(ha), wa) == lib.FSE_readNCount(xb, C.byref(m2), C.byref(t2), ptr(hb), wb)
        assert (m1.value, t1.value) == (m2.value, t2.value) and list(xa)[:msv + 1] == list(xb)[:msv + 1]
        cta = np.zeros(1 + 2048 + 512, np.uint32); ctb = np.zeros_like(cta)
        assert g_ct(ptr(cta), na, msv, tl) == lib.FSE_buildCTable(ptr(ctb), nb_, msv, tl) == 0
        half = 1 + (1 << (tl - 1))
        assert np.array_equal(cta[:half], ctb[:half])
        for s in range(msv + 1):
            assert cta[half + 2 * s + 1] == ctb[half + 2 * s + 1]
            if na[s] != 0:
                assert cta[half + 2 * s] == ctb[half + 2 * s]
        dta = np.zeros(1 + 4096, np.uint32); dtb = np.zeros_like(dta)
        assert g_dt(ptr(dta), na, msv, tl) == lib.FSE_buildDTable(ptr(dtb), nb_, msv, tl) == 0
        assert np.array_equal(dta[:1 + (1 << tl)], dtb[:1 + (1 << tl)])
        # Huffman side
        hl = lib.HUF_optimalTableLog(12, n, msv)
        ta = np.zeros(256, np.uint32); tb = np.zeros(256, np.uint32)
        r1 = g_hct(ptr(ta), ca, msv, hl); r2 = lib.HUF_buildCTable(ptr(tb), cb, msv, hl)
        assert r1 == r2 and np.array_equal(ta[:msv + 1] & 0xFFFFFF, tb[:msv + 1] & 0xFFFFFF)
        ha = np.zeros(300, np.uint8); hb = np.zeros(300, np.uint8)
        wa = g_hw(ptr(ha), 300, ptr(ta), msv, r1); wb = lib.HUF_writeCTable(ptr(hb), 300, ptr(tb), msv, r2)
        assert wa == wb
        if is_error(wa):
            continue
        assert bytes(ha[:wa]) == bytes(hb[:wb])
        wA = np.zeros(260, np.uint8); wB = np.zeros(260, np.uint8); rsA = (C.c_uint32 * 17)(); rsB = (C.c_uint32 * 17)()
        nA, nB, tA, tB = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
        sa = g_hrs(ptr(wA), 256, rsA, C.byref(nA), C.byref(tA), ptr(ha), wa)
        sb = lib.HUF_readStats(ptr(wB), 256, rsB, C.byref(nB), C.byref(tB), ptr(hb), wb)
        assert sa == sb
        if is_error(sa):
            continue
        assert (nA.value, tA.value) == (nB.value, tB.value) and bytes(wA[:nA.value]) == bytes(wB[:nB.value]) and list(rsA)[:13] == list(rsB)[:13]
        dA = np.zeros(1 + 2048, np.uint32); dB = np.zeros(1 + 2048, np.uint32); dA[0] = dB[0] = 11 * 0x01000001
        assert g_hdt(ptr(dA), ptr(ha), wa) == lib.HUF_readDTableX1(ptr(dB), ptr(hb), wb) == wa
        ncell = 1 + ((1 << tA.value) + 1) // 2
        assert np.array_equal(dA[:ncell], dB[:ncell])
        # payload coding with the caller's tables: FSE_compress_usingCTable / FSE_decompress_usingDTable /
        # HUF_compress4X_usingCTable / HUF_decompress4X[1]_usingDTable (same images on both sides)
        g_euc = sig("FSE_compress_usingCTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
        g_dud = sig("FSE_decompress_usingDTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
        g_huc = sig("HUF_compress4X_usingCTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
        g_hud = sig("HUF_decompress4X_usingDTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
        for r_ in ("FSE_compress_usingCTable", "FSE_decompress_usingDTable", "HUF_compress4X_usingCTable", "HUF_decompress4X_usingDTable"):
            f = getattr(lib, r_); f.restype = C.c_size_t; f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
        for cap in (n + 600, max(16, n // 3)):
            oa = np.zeros(cap + 16, np.uint8); ob = np.zeros(cap + 16, np.uint8)
            ea = g_euc(ptr(oa), cap, ptr(d), n, ptr(ctb)); eb = lib.FSE_compress_usingCTable(ptr(ob), cap, ptr(d), n, ptr(ctb))
            assert ea == eb and bytes(oa[:ea]) == bytes(ob[:eb])
            if ea and cap > n:
                ra_ = np.zeros(n + 8, np.uint8); rb_ = np.zeros(n + 8, np.uint8)
                for dcap in (n, n - 1, n + 5):
                    da = g_dud(ptr(ra_), dcap, ptr(oa), ea, ptr(dtb)); db = lib.FSE_decompress_usingDTable(ptr(rb_), dcap, ptr(ob), eb, ptr(dtb))
                    assert da == db
                    if not is_error(da):
                        assert bytes(ra_[:da]) == bytes(rb_[:db])
                bad = oa[:ea].copy(); bad[int(rng.integers(0, ea))] ^= 1 << int(rng.integers(0, 8))
                da = g_dud(ptr(ra_), n, ptr(bad), ea, ptr(dtb)); db = lib.FSE_decompress_usingDTable(ptr(rb_), n, ptr(bad), ea, ptr(dtb))
                assert da == db
            ha2 = np.zeros(cap + 16, np.uint8); hb2 = np.zeros(cap + 16, np.uint8)
            ea = g_huc(ptr(ha2), cap, ptr(d), n, ptr(tb)); eb = lib.HUF_compress4X_usingCTable(ptr(hb2), cap, ptr(d), n, ptr(tb))
            assert ea == eb and bytes(ha2[:ea]) == bytes(hb2[:eb])
            if ea and n >= 6:
                ra_ = np.zeros(n + 8, np.uint8); rb_ = np.zeros(n + 8, np.uint8)
                da = g_hud(ptr(ra_), n, ptr(ha2), ea, ptr(dB)); db = lib.HUF_decompress4X_usingDTable(ptr(rb_), n, ptr(hb2), eb, ptr(dB))
                assert da == db == n and bytes(ra_[:n]) == bytes(rb_[:n]) == bytes(d[:n])
                bad = ha2[:ea].copy(); bad[int(rng.integers(6, ea))] ^= 1 << int(rng.integers(0, 8))      # past the jump table: the CPU library trusts it
                da = g_hud(ptr(ra_), n, ptr(bad), ea, ptr(dB)); db = lib.HUF_decompress4X_usingDTable(ptr(rb_), n, ptr(bad), ea, ptr(dB))
                assert is_error(da) == is_error(db)
                if is_error(da):
                    assert da == db


@pytest.mark.parametrize("codec,p,mib", [("huf", 0.14, 64), ("fse", 0.80, 16)])
def test_large_roundtrip_property(codec, p, mib):
    """BASELINE sizes are too big for the CPU checker in a test: use encode -> decode == identity, a
    checksum of per-block sizes against a CPU sample, and the GPU<->CPU cross-decode on that sample"""
    n = mib << 20
    data = probagen(n, p)
    d = _dev(data)
    cbuf, cs = ENC[codec](d, BLOCK, SLOT, 255, 12)
    out, res = DEC[codec](cbuf, cs, n, BLOCK, SLOT, orig=d)
    torch.cuda.synchronize()
    assert torch.equal(out, d)
    assert bool((res == BLOCK).all())
    sample = slice(0, 64 * BLOCK)
    wc, wcs, _ = cpu_compress(codec, data[sample], slot=SLOT)
    assert np.array_equal(cs[:64].cpu().numpy().view(np.uint64), wcs)
    got = cbuf[:64 * SLOT].cpu().numpy()
    for b in range(64):
        assert np.array_equal(got[b * SLOT: b * SLOT + int(wcs[b])], wc[b * SLOT: b * SLOT + int(wcs[b])])


@pytest.mark.parametrize("codec,mib", [("huf", 256), ("fse", 256), ("u16", 256)])
def test_full_compare_at_256mib(codec, mib):
    """BASELINE configs[1] / [2] / [4] at 256 MiB: EVERY block's return value and compressed bytes against the compiled reference
    (its pthread block loop, oracle/ref_shim.c), the GPU decoding the reference's blocks, and the identity round trip."""
    lib, isref = checker()
    n = mib << 20
    if codec == "u16":
        data = gen_u16(n // 2, 240, 0.50, 1).view(np.uint8); slot, msv, tl = 32768, 0, 12
    else:
        data = probagen(n, 0.14 if codec == "huf" else 0.80); slot, msv, tl = SLOT, 255, 12
    nb = n // BLOCK
    wc, wcs, _ = cpu_compress(codec, data, slot=slot, msv=msv, tl=tl)
    d = _dev(data)
    cbuf, cs = ENC[codec](d, BLOCK, slot, msv, tl)
    out, res = DEC[codec](cbuf, cs, n, BLOCK, slot, orig=d)
    o2, r2 = DEC[codec](_dev(wc), _dev(wcs), n, BLOCK, slot, orig=d)        # the reference's blocks through our decoder
    torch.cuda.synchronize()
    assert torch.equal(out, d) and torch.equal(o2, d)
    assert np.array_equal(cs.cpu().numpy().view(np.uint64), wcs)
    got = cbuf[:nb * slot].cpu().numpy().reshape(nb, slot); want = wc[:nb * slot].reshape(nb, slot)
    sizes = wcs.astype(np.int64); sizes[wcs > np.uint64(1 << 62)] = 0
    if codec != "huf":
        sizes[sizes == 1] = 0
    cols = np.arange(slot, dtype=np.int64)[None, :]
    for c0 in range(0, nb, 1024):
        bad = (got[c0:c0 + 1024] != want[c0:c0 + 1024]) & (cols < sizes[c0:c0 + 1024, None])
        assert not bad.any(), (codec, c0 + int(np.argwhere(bad)[0][0]))
    assert int(sizes.sum()) > n // 20


def test_raw_and_rle_tables_through_payload_calls():
    """FSE_buildCTable_raw/_rle + FSE_buildDTable_raw/_rle images driven through FSE_compress_usingCTable /
    FSE_decompress_usingDTable on the GPU vs the compiled reference (fullbench.c:595-629 call pattern)"""
    lib, isref = checker()
    L = fb.lib()
    def sig(M, n, *a):
        f = getattr(M, n); f.restype = C.c_size_t; f.argtypes = list(a); return f
    for M in (L, lib):
        sig(M, "FSE_buildCTable_raw", C.c_void_p, U); sig(M, "FSE_buildDTable_raw", C.c_void_p, U)
        sig(M, "FSE_buildCTable_rle", C.c_void_p, C.c_ubyte); sig(M, "FSE_buildDTable_rle", C.c_void_p, C.c_ubyte)
        sig(M, "FSE_compress_usingCTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
        sig(M, "FSE_decompress_usingDTable", C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p)
    rng = np.random.default_rng(77)
    for nb in (1, 3, 6, 8):
        n = int(rng.integers(50, 5000))
        d = rng.integers(0, 1 << nb, n, dtype=np.uint8)
        ct = np.zeros(1 + 128 + 2 * 256 + 8, np.uint32); dt = np.zeros(1 + 256 + 8, np.uint32)
        assert L.FSE_buildCTable_raw(ptr(ct), nb) == 0 and L.FSE_buildDTable_raw(ptr(dt), nb) == 0
        cap = n + 64
        oa = np.zeros(cap + 16, np.uint8); ob = np.zeros(cap + 16, np.uint8)
        ea = L.FSE_compress_usingCTable(ptr(oa), cap, ptr(d), n, ptr(ct)); eb = lib.FSE_compress_usingCTable(ptr(ob), cap, ptr(d), n, ptr(ct))
        assert ea == eb and bytes(oa[:ea]) == bytes(ob[:eb])
        if ea:
            ra = np.zeros(n + 8, np.uint8); rb = np.zeros(n + 8, np.uint8)
            da = L.FSE_decompress_usingDTable(ptr(ra), n, ptr(oa), ea, ptr(dt)); db = lib.FSE_decompress_usingDTable(ptr(rb), n, ptr(ob), eb, ptr(dt))
            assert da == db == n and bytes(ra[:n]) == bytes(rb[:n]) == bytes(d)
    for sym in (0, 200):
        n = 777
        d = np.full(n, sym, np.uint8)
        ct = np.zeros(2 + 2 * 256 + 8, np.uint32); dt = np.zeros(4, np.uint32)
        assert L.FSE_buildCTable_rle(ptr(ct), sym) == 0 and L.FSE_buildDTable_rle(ptr(dt), sym) == 0
        oa = np.zeros(128, np.uint8); ob = np.zeros(128, np.uint8)
        ea = L.FSE_compress_usingCTable(ptr(oa), 100, ptr(d), n, ptr(ct)); eb = lib.FSE_compress_usingCTable(ptr(ob), 100, ptr(d), n, ptr(ct))
        assert ea == eb and bytes(oa[:ea]) == bytes(ob[:eb])


def test_single_stream_huff0():
    """HUF_compress1X / HUF_compress1X_usingCTable / HUF_decompress1X1 / HUF_decompress1X_usingDTable vs the compiled reference"""
    lib, isref = checker()
    L = fb.lib()
    for M in (L, lib):
        for n_, a_ in (("HUF_compress1X", [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, U, U]),
                       ("HUF_decompress1X1", [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
                       ("HUF_compress1X_usingCTable", [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
                       ("HUF_buildCTable", [C.c_void_p, C.c_void_p, U, U]),
                       ("HIST_count", [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t])):
            f = getattr(M, n_); f.restype = C.c_size_t; f.argtypes = a_
    rng = np.random.default_rng(91)
    for it in range(14):
        n = int(rng.integers(1, 30000)) if it else 20000
        d = zoo(rng, n)
        for cap in (n + 300, max(1, n // 2)):
            oa = np.zeros(cap + 16, np.uint8); ob = np.zeros(cap + 16, np.uint8)
            ea = L.HUF_compress1X(ptr(oa), cap, ptr(d), n, 255, 11); eb = lib.HUF_compress1X(ptr(ob), cap, ptr(d), n, 255, 11)
            assert ea == eb, (it, n, cap, ea, eb)
            if is_error(ea) or ea <= 1:
                continue
            assert bytes(oa[:ea]) == bytes(ob[:eb])
            ra = np.zeros(n + 8, np.uint8); rb = np.zeros(n + 8, np.uint8)
            da = L.HUF_decompress1X1(ptr(ra), n, ptr(oa), ea); db = lib.HUF_decompress1X1(ptr(rb), n, ptr(ob), eb)
            assert da == db == n and bytes(ra[:n]) == bytes(d[:n])
            bad = oa[:ea].copy(); bad[int(rng.integers(0, ea))] ^= 1 << int(rng.integers(0, 8))
            da = L.HUF_decompress1X1(ptr(ra), n, ptr(bad), ea); db = lib.HUF_decompress1X1(ptr(rb), n, ptr(bad), ea)
            assert da == db
        # payload only, with the reference's own table
        cnt = (U * 256)(); m = U(255)
        if is_error(lib.HIST_count(cnt, C.byref(m), ptr(d), n)) or m.value == 0:
            continue
        ct = np.zeros(256, np.uint32)
        if is_error(lib.HUF_buildCTable(ptr(ct), cnt, m.value, 11)):
            continue
        oa = np.zeros(n + 300, np.uint8); ob = np.zeros(n + 300, np.uint8)
        ea = L.HUF_compress1X_usingCTable(ptr(oa), n + 256, ptr(d), n, ptr(ct)); eb = lib.HUF_compress1X_usingCTable(ptr(ob), n + 256, ptr(d), n, ptr(ct))
        assert ea == eb and bytes(oa[:ea]) == bytes(ob[:eb])


def test_double_symbol_table_and_decoders():
    """HUF_readDTableX2 image (a18) word-equal with the reference at maxTableLog 11 and 12, and HUF_decompress4X2/1X2/4X/1X
    _usingDTable on that image vs the reference, valid and bit-flipped streams"""
    lib, isref = checker()
    L = fb.lib()
    S = C.c_size_t; V = C.c_void_p
    for M in (L, lib):
        for n_, a_ in (("HUF_readDTableX2", [V, V, S]), ("HUF_decompress4X2_usingDTable", [V, S, V, S, V]), ("HUF_decompress1X2_usingDTable", [V, S, V, S, V]),
                       ("HUF_decompress4X_usingDTable", [V, S, V, S, V]), ("HUF_decompress1X_usingDTable", [V, S, V, S, V]),
                       ("HUF_compress4X_usingCTable", [V, S, V, S, V]), ("HUF_compress1X_usingCTable", [V, S, V, S, V]),
                       ("HUF_buildCTable", [V, V, U, U]), ("HUF_writeCTable", [V, S, V, U, U]), ("HIST_count", [V, V, V, S])):
            f = getattr(M, n_); f.restype = S; f.argtypes = a_
    lib.HUF_optimalTableLog.argtypes = [U, S, U]
    rng = np.random.default_rng(313)
    done = 0
    for it in range(40):
        n = int(rng.integers(400, 40000)); d = zoo(rng, n)
        cnt = (U * 256)(); m = U(255)
        mx = lib.HIST_count(cnt, C.byref(m), ptr(d), n)
        if is_error(mx) or mx == n or m.value == 0:
            continue
        msv = m.value
        ct = np.zeros(256, np.uint32)
        hl = lib.HUF_buildCTable(ptr(ct), cnt, msv, lib.HUF_optimalTableLog(11, n, msv))
        if is_error(hl):
            continue
        hdr = np.zeros(300, np.uint8)
        hs = lib.HUF_writeCTable(ptr(hdr), 300, ptr(ct), msv, hl)
        if is_error(hs):
            continue
        for Lg in (12, 11):
            xa = np.zeros(1 + 4096, np.uint32); xb = np.zeros(1 + 4096, np.uint32); xa[0] = xb[0] = Lg * 0x01000001
            qa = L.HUF_readDTableX2(ptr(xa), ptr(hdr), hs); qb = lib.HUF_readDTableX2(ptr(xb), ptr(hdr), hs)
            assert qa == qb, (it, Lg, qa, qb)
            if is_error(qa):
                continue
            assert np.array_equal(xa[:1 + (1 << Lg)], xb[:1 + (1 << Lg)]), (it, Lg)
            for enc, deca, decb in ((lib.HUF_compress4X_usingCTable, L.HUF_decompress4X2_usingDTable, lib.HUF_decompress4X2_usingDTable),
                                    (lib.HUF_compress1X_usingCTable, L.HUF_decompress1X2_usingDTable, lib.HUF_decompress1X2_usingDTable),
                                    (lib.HUF_compress4X_usingCTable, L.HUF_decompress4X_usingDTable, lib.HUF_decompress4X_usingDTable),
                                    (lib.HUF_compress1X_usingCTable, L.HUF_decompress1X_usingDTable, lib.HUF_decompress1X_usingDTable)):
                cb = np.zeros(n + 600, np.uint8)
                e = enc(ptr(cb), n + 512, ptr(d), n, ptr(ct))
                if is_error(e) or e == 0:
                    continue
                oa = np.zeros(n + 16, np.uint8); ob = np.zeros(n + 16, np.uint8)
                ra = deca(ptr(oa), n, ptr(cb), e, ptr(xb)); rb = decb(ptr(ob), n, ptr(cb), e, ptr(xb))
                assert ra == rb == n and bytes(oa[:n]) == bytes(d[:n]), (it, Lg, ra, rb)
                bad = cb[:e].copy(); bad[int(rng.integers(6, e))] ^= 1 << int(rng.integers(0, 8))
                ra = deca(ptr(oa), n, ptr(bad), e, ptr(xb)); rb = decb(ptr(ob), n, ptr(bad), e, ptr(xb))
                assert is_error(ra) == is_error(rb)
                done += 1
    assert done > 20
