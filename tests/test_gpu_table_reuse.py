"""SURVEY.md section 8f-3: Huffman table reuse across blocks, against the compiled reference's recorded calls (-m gpu).

  * FSEB200_HUF_compress4X_usingCTable_batch : every block of a batch coded with ONE table == the reference's
    HUF_compress4X_usingCTable per block (lib/huf.h:191), bytes and return values, incl. blocks the table does not cover well,
    short / ragged blocks and undersized slots;
  * HUF_compress4X_repeat / HUF_compress1X_repeat (lib/huf.h:204,296; huf_compress.c:637-724) as a SEQUENCE of calls that carries
    (table, repeat flag) from block to block, for every starting flag and preferRepeat value;
  * HUF_readCTable round trip (lib/huf.h:231)."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import load_ref, ptr, zoo, probagen, is_error
import finitestateentropy_b200 as fb

pytestmark = pytest.mark.gpu
S, V, U = C.c_size_t, C.c_void_p, C.c_uint


def _libs():
    ref = load_ref()
    L = fb.lib()
    for X in (L, ref):
        X.HUF_compress4X_repeat.restype = S
        X.HUF_compress4X_repeat.argtypes = [V, S, V, S, U, U, V, S, V, C.POINTER(C.c_int), C.c_int, C.c_int]
        X.HUF_compress1X_repeat.restype = S
        X.HUF_compress1X_repeat.argtypes = [V, S, V, S, U, U, V, S, V, C.POINTER(C.c_int), C.c_int, C.c_int]
        X.HUF_readCTable.restype = S
        X.HUF_readCTable.argtypes = [V, C.POINTER(U), V, S, C.POINTER(U)]
    L.FSEB200_HUF_compress4X_usingCTable_batch.restype = S
    L.FSEB200_HUF_compress4X_usingCTable_batch.argtypes = [V, S, V, V, S, S, V, V]
    return L, ref


def _ref_table(ref, data):
    cnt = (U * 256)(); m = U(255)
    ref.HIST_count(cnt, C.byref(m), ptr(data), len(data))
    ct = np.zeros(256, np.uint32)
    tl = ref.HUF_optimalTableLog(12, len(data), m.value)
    r = ref.HUF_buildCTable(ptr(ct), cnt, m.value, tl)
    assert not is_error(r)
    return ct


def test_batch_with_one_table_matches_the_reference_block_by_block():
    L, ref = _libs()
    rng = np.random.default_rng(31)
    for block, slot in ((32768, 33548), (4099, 4700), (1000, 600), (12, 64), (11, 64)):
        parts = [probagen(block * 20, 0.14), probagen(block * 6, 0.30), zoo(rng, block * 3), np.full(block * 2, 9, np.uint8), probagen(int(rng.integers(1, block)), 0.14)]
        data = np.concatenate(parts)
        ct = _ref_table(ref, probagen(65536, 0.14) if block >= 12 else data)   # table of the dominant distribution; other blocks fit it badly or not at all
        nb = (len(data) + block - 1) // block
        want_c = np.zeros(nb * slot + 64, np.uint8); want = np.zeros(nb, np.uint64)
        for b in range(nb):
            blk = np.ascontiguousarray(data[b * block:(b + 1) * block])
            want[b] = ref.HUF_compress4X_usingCTable(ptr(want_c[b * slot:]), slot, ptr(blk), len(blk), ptr(ct))
        d_src = torch.from_numpy(data).cuda(); d_ct = torch.from_numpy(ct.view(np.int32)).cuda()
        d_c = torch.zeros(nb * slot + 64, dtype=torch.uint8, device="cuda"); d_s = torch.zeros(nb, dtype=torch.int64, device="cuda")
        r = L.FSEB200_HUF_compress4X_usingCTable_batch(d_c.data_ptr(), slot, d_s.data_ptr(), d_src.data_ptr(), len(data), block, d_ct.data_ptr(),
                                                       torch.cuda.current_stream().cuda_stream)
        assert r == 0
        torch.cuda.synchronize()
        got = d_s.cpu().numpy().view(np.uint64); got_c = d_c.cpu().numpy()
        assert np.array_equal(got, want), (block, [(int(a), int(b)) for a, b in zip(got, want) if a != b][:5])
        for b in range(nb):
            k = int(want[b])
            assert np.array_equal(got_c[b * slot:b * slot + k], want_c[b * slot:b * slot + k]), (block, b)
        assert (want > 1).sum() >= (3 if block >= 1000 else 0)


@pytest.mark.parametrize("four", [True, False])
def test_repeat_sequences_carry_table_and_flag_like_the_reference(four):
    L, ref = _libs()
    rng = np.random.default_rng(32)
    name = "HUF_compress4X_repeat" if four else "HUF_compress1X_repeat"
    for start_flag in (0, 1, 2):
        for prefer in (0, 1):
            blocks = [probagen(20000, 0.14), probagen(20000, 0.14)[5000:], probagen(9000, 0.3), zoo(rng, 7000), np.full(3000, 5, np.uint8),
                      rng.integers(0, 256, 4000, dtype=np.uint8), probagen(30000, 0.2), probagen(100, 0.14), probagen(30000, 0.2)[100:]]
            ta = _ref_table(ref, probagen(40000, 0.14)); tb = ta.copy()
            fa = C.c_int(start_flag); fb_ = C.c_int(start_flag)
            wa = np.zeros(2048, np.uint32); wb = np.zeros(2048, np.uint32)
            for i, d in enumerate(blocks):
                d = np.ascontiguousarray(d); n = len(d); cap = n + 600
                oa = np.zeros(cap + 8, np.uint8); ob = np.zeros(cap + 8, np.uint8)
                ra = getattr(L, name)(ptr(oa), cap, ptr(d), n, 255, 11, ptr(wa), wa.nbytes, ptr(ta), C.byref(fa), prefer, 0)
                rb = getattr(ref, name)(ptr(ob), cap, ptr(d), n, 255, 11, ptr(wb), wb.nbytes, ptr(tb), C.byref(fb_), prefer, 0)
                assert ra == rb, (start_flag, prefer, i, ra, rb)
                assert fa.value == fb_.value and np.array_equal(ta, tb), (start_flag, prefer, i)
                if not is_error(ra) and ra > 1:
                    assert np.array_equal(oa[:ra], ob[:rb]), (start_flag, prefer, i)
                if i == 4:                                              # a caller marks the table "to be checked" again, as zstd does between frames
                    fa.value = fb_.value = 1


def test_read_ctable_round_trip():
    L, ref = _libs()
    for p in (0.14, 0.3, 0.02, 0.8):
        d = probagen(32768, p)
        ct = _ref_table(ref, d)
        cnt = (U * 256)(); m = U(255); ref.HIST_count(cnt, C.byref(m), ptr(d), len(d))
        nbits = (ct >> 16) & 0xFF
        hdr = np.zeros(256, np.uint8)
        h = ref.HUF_writeCTable(ptr(hdr), 256, ptr(ct), m.value, int(nbits[:m.value + 1].max()))
        assert not is_error(h)
        for X in (L, ref):
            out = np.zeros(256, np.uint32); msv = U(255); hz = U(9)
            r = X.HUF_readCTable(ptr(out), C.byref(msv), ptr(hdr), h, C.byref(hz))
            assert r == h and msv.value == m.value
            assert np.array_equal(out[:m.value + 1] & 0x00FFFFFF, ct[:m.value + 1] & 0x00FFFFFF), p
