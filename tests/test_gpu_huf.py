"""Parity of the CUDA Huff0 path against the CPU checker, through the C-ABI (-m gpu)."""
import ctypes as C
import numpy as np
import pytest
import torch

from helpers import load_port, ptr, zoo, rand_size, probagen, is_error
from gpu_common import cpu_compress, cpu_decompress, checker, BLOCK, SLOT
import finitestateentropy_b200 as fb

pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8) if a.dtype != np.uint64 else a.view(np.int64)).cuda()


def _decode_and_check(data, block, cbuf, cs, slot, orig_for_raw=True):
    d_c = _dev(cbuf); d_s = _dev(cs)
    d_o = _dev(data) if orig_for_raw else None
    out, res = fb.huf_decompress_batch(d_c, d_s, len(data), block, slot, orig=d_o)
    torch.cuda.synchronize()
    res = res.cpu().numpy().view(np.uint64)
    out = out.cpu().numpy()
    nb = (len(data) + block - 1) // block
    # expected verdicts from the CPU checker (a 1-bit code at tableLog 12 is undecodable for the reference itself)
    want_out, want = cpu_decompress("huf", cbuf, cs, data, block=block, slot=slot)
    for b in range(nb):
        n = min(block, len(data) - b * block)
        assert res[b] == want[b], (b, int(res[b]), int(want[b]), n, int(cs[b]))
        if not is_error(int(want[b])):
            assert res[b] == n
            assert np.array_equal(out[b * block: b * block + n], data[b * block: b * block + n]), b
    assert sum(1 for b in range(nb) if not is_error(int(want[b]))) > nb // 2


@pytest.mark.parametrize("p", [0.14, 0.20, 0.80, 0.02])
def test_decode_probagen_1mib(p):
    data = probagen(1048575, p)                      # programs/probaGenerator.c:47 size, 32 blocks, last one 32767
    cbuf, cs, slot = cpu_compress("huf", data)
    assert (cs > 1).all()
    _decode_and_check(data, BLOCK, cbuf, cs, slot)


def test_decode_zoo_ragged_blocks():
    """every block shape the fuzzers use, incl. raw (0), RLE (1), tiny and non-multiple-of-4 sizes"""
    rng = np.random.default_rng(11)
    for block in (32768, 4099, 1000, 131072, 12, 77):
        parts = [zoo(rng, block) for _ in range(int(rng.integers(3, 70)))]
        parts.append(zoo(rng, int(rng.integers(1, block + 1))))
        data = np.concatenate(parts)
        cbuf, cs, slot = cpu_compress("huf", data, block=block)
        _decode_and_check(data, block, cbuf, cs, slot)


def _corrupt_blocks(rng, data, block, count_modes=3):
    cbuf, cs, slot = cpu_compress("huf", data, block=block)
    for b in range(len(cs)):
        if cs[b] < 2:
            continue
        c = cbuf[b * slot: b * slot + int(cs[b])]
        mode = int(rng.integers(0, count_modes))
        if mode == 0:
            cs[b] = int(rng.integers(2, int(cs[b])))
        elif mode == 1:
            for _ in range(int(rng.integers(1, 4))):
                c[int(rng.integers(0, len(c)))] ^= int(rng.integers(1, 256))
    return cbuf, cs, slot


def test_decode_error_verdicts():
    """truncated / bit-flipped blocks through the batch call: the verdict AND the bytes of the reference's HUF_decompress
    (which runs X1 or X2 as HUF_selectDecoder says -- X2 accepts streams X1 rejects), nothing written past the batch"""
    lib, isref = checker()
    dec = lib.HUF_decompress if isref else lib.orc_huf_decompress
    dec_x1 = lib.HUF_decompress4X1 if isref else lib.orc_huf_decompress4x1
    rng = np.random.default_rng(12)
    x2_only = 0
    for block in (8192, 32768):
        data = np.concatenate([zoo(rng, block) if i % 3 else probagen(block, [0.14, 0.2, 0.3][i % 9 // 3]) for i in range(200)])
        cbuf, cs, slot = _corrupt_blocks(rng, data, block)
        nb = len(cs)
        want = np.zeros(nb, np.uint64); want_out = np.zeros(len(data), np.uint8)
        for b in range(nb):
            if cs[b] < 2:
                want[b] = block; want_out[b * block:(b + 1) * block] = data[b * block:(b + 1) * block]
                continue
            tmp = np.concatenate([cbuf[b * slot: b * slot + int(cs[b])], np.zeros(32, np.uint8)])
            o = np.zeros(block + 8, np.uint8)
            want[b] = dec(ptr(o), block, ptr(tmp), int(cs[b]))
            want_out[b * block:(b + 1) * block] = o[:block]
            if not is_error(int(want[b])) and cs[b] != block:
                o2 = np.zeros(block + 8, np.uint8)
                x2_only += bool(is_error(dec_x1(ptr(o2), block, ptr(tmp), int(cs[b]))))
        guard = torch.full((len(data) + 4096,), 0x5A, dtype=torch.uint8, device="cuda")
        out, res = fb.huf_decompress_batch(_dev(cbuf), _dev(cs), len(data), block, slot, out=guard, orig=_dev(data))
        torch.cuda.synchronize()
        res = res.cpu().numpy().view(np.uint64); out = out.cpu().numpy()
        bad = [(b, int(res[b]), int(want[b])) for b in range(nb) if res[b] != want[b]]
        assert not bad, bad[:10]
        for b in range(nb):
            if not is_error(int(want[b])):
                assert np.array_equal(out[b * block:(b + 1) * block], want_out[b * block:(b + 1) * block]), b
        assert (guard[len(data):] == 0x5A).all()
        assert sum(is_error(int(x)) for x in want) > 10
    assert x2_only > 0          # the sweep contains streams that only the double-symbol decoder accepts


def test_fixed_decoder_entry_points_on_corrupted_blocks():
    """HUF_decompress / HUF_decompress4X1 / HUF_decompress4X2 (host pointers): each returns its CPU namesake's value and bytes"""
    lib, isref = checker()
    L = fb.lib()
    for nm in ("HUF_decompress", "HUF_decompress4X1", "HUF_decompress4X2"):
        f = getattr(L, nm); f.restype = C.c_size_t; f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    rng = np.random.default_rng(14)
    block = 32768
    data = np.concatenate([probagen(block, p) for p in (0.14, 0.2, 0.14, 0.3, 0.14, 0.2) * 10])
    cbuf, cs, slot = _corrupt_blocks(rng, data, block)
    disagree = 0
    for b in range(len(cs)):
        if cs[b] < 2 or cs[b] >= block:
            continue
        tmp = np.concatenate([cbuf[b * slot: b * slot + int(cs[b])], np.zeros(32, np.uint8)])
        vals = {}
        for nm in ("HUF_decompress", "HUF_decompress4X1", "HUF_decompress4X2"):
            oa = np.full(block + 8, 0x33, np.uint8); ob = np.full(block + 8, 0x33, np.uint8)
            ra = getattr(L, nm)(ptr(oa), block, ptr(tmp), int(cs[b]))
            rb = getattr(lib, nm)(ptr(ob), block, ptr(tmp), int(cs[b]))
            assert ra == rb, (b, nm, ra, rb)
            assert (oa[block:] == 0x33).all()
            if not is_error(ra):
                assert np.array_equal(oa, ob), (b, nm)
            vals[nm] = ra
        disagree += vals["HUF_decompress4X1"] != vals["HUF_decompress4X2"]
    assert disagree > 0


def test_single_block_host_api():
    """the reference-named one-block entry point with host pointers (lib/huf.h:67)"""
    L = fb.lib()
    rng = np.random.default_rng(13)
    for n in (32768, 1000, 70000, 13):
        d = zoo(rng, n) if n != 13 else np.arange(13, dtype=np.uint8) % 3
        cbuf, cs, slot = cpu_compress("huf", d, block=n)
        if cs[0] < 2:
            continue
        out = np.zeros(n, np.uint8)
        r = L.HUF_decompress(ptr(out), n, ptr(cbuf), int(cs[0]))
        assert r == n and np.array_equal(out, d)
