"""Oracle port against the committed golden vectors (tests/golden/, generated from the compiled
reference by make_golden.py) and the known-answer values recorded in SURVEY.md section 6.3.
CPU only; needs neither /root/reference nor oracle/_ref."""
import hashlib
import json
import os

import numpy as np

from helpers import load_port, ptr, probagen, gen_u16, is_error, small_vectors, sha256

HERE = os.path.dirname(os.path.abspath(__file__))
KATS = json.load(open(os.path.join(HERE, "golden", "kat_bench.json")))
BLOCK, SLOT = 32768, 33548

# SURVEY.md section 6.3 (values extracted from the reference by the survey, independent of make_golden.py)
SURVEY_63 = {
    ("proba20", "fse"): (474361, "b58c28d0fed570b5"), ("proba20", "huf"): (478076, "65a7281774f18f77"),
    ("proba14", "fse"): (548948, "20a2e94b87d046b9"), ("proba14", "huf"): (552203, "facfb967534afdaf"),
    ("proba80", "fse"): (118641, "d5edf7868e6b7acd"), ("proba80", "huf"): (164244, "8786e43b17bc582a"),
    ("proba02", "fse"): (928392, "9d083be4c87118cd"), ("proba02", "huf"): (926583, "856cbaf271878cab"),
    ("u16_p50", "u16"): (131685, "b85fe0fce48c4f25"),
}
SURVEY_MD5 = {"proba20": "6b271f552ee8128578ea3fb0b6b3ac43", "proba14": "ac6f59cd6545e7a44aa362832ec8da2b",
              "proba80": "7eadfac6f83805f07fdf9345fba9d673", "proba02": "7b73bf489a99e28828b6667f23927baa"}


def _input(name):
    if name == "u16_p50":
        return gen_u16(524288, 240, 0.50, 1).view(np.uint8)
    return probagen(1048575, int(name[5:]) / 100.0)


def test_generators_match_reference_md5():
    for name, md5 in SURVEY_MD5.items():
        assert hashlib.md5(_input(name).tobytes()).hexdigest() == md5
    port = load_port()
    u = gen_u16(524288, 240, 0.50, 1)
    assert "%016x" % port.orc_xxh64(ptr(u), u.nbytes, 0) == "deb703351ea4b547"      # SURVEY.md 6.3, U16 row
    big = probagen(3 * 1048575 + 17, 0.14)                                             # prefix stability
    assert hashlib.md5(big[:1048575].tobytes()).hexdigest() == SURVEY_MD5["proba14"]


def test_kat_bench_runs():
    port = load_port()
    for rec in KATS:
        data = np.ascontiguousarray(_input(rec["name"]))
        assert hashlib.md5(data.tobytes()).hexdigest() == rec["srcMd5"]
        nb = (len(data) + BLOCK - 1) // BLOCK
        cbuf = np.zeros(nb * SLOT, np.uint8)
        cs = np.zeros(nb, np.uint64)
        codec = {"fse": 0, "huf": 1, "u16": 2}[rec["codec"]]
        slot = 32768 if codec == 2 else SLOT
        port.orc_compress_blocks(codec, ptr(data), len(data), BLOCK, ptr(cbuf), slot, ptr(cs), rec["maxSymbolValue"], rec["tableLog"])
        assert [int(x) for x in cs] == rec["cSizes"]
        cat = np.concatenate([cbuf[b * slot: b * slot + int(cs[b])] for b in range(nb)])
        h = "%016x" % port.orc_xxh64(ptr(cat), len(cat), 0)
        assert h == rec["xxh64"]
        assert (rec["total"], rec["xxh64"]) == SURVEY_63[(rec["name"], rec["codec"])]
        out = np.zeros(len(data), np.uint8); res = np.zeros(nb, np.uint64)
        port.orc_decompress_blocks(codec, ptr(out), ptr(data), len(data), BLOCK, ptr(cbuf), slot, ptr(cs), ptr(res))
        assert np.array_equal(out, data)
        assert port.orc_xxh32(ptr(out), len(out), 0) == port.orc_xxh32(ptr(data), len(data), 0)   # bench.c:311,444


def test_small_vectors():
    port = load_port()
    z = np.load(os.path.join(HERE, "golden", "vectors_small.npz"))
    kinds = set()
    vecs = list(small_vectors())
    assert len(vecs) == int(z["count"][0])
    for k, (codec, d) in enumerate(vecs):
        assert codec == int(z["codec"][k]) and sha256(d) == z["in_sha256"][k], k      # the recorded input
        want = int(z["ret"][k])
        n = len(d)
        if codec == 2:
            dst = np.zeros(n + 600, np.uint8)
            r = port.orc_fse_compress_u16(ptr(dst), n + 592, ptr(d), n // 2, 0, 12)
        else:
            cap = 512 + n + (n >> 7) + 12
            dst = np.zeros(cap + 8, np.uint8)
            r = (port.orc_fse_compress2 if codec == 0 else port.orc_huf_compress2)(ptr(dst), cap, ptr(d), n, 255, 12)
        assert r == want, (k, codec, n, r, want)
        kinds.add("err" if is_error(r) else min(r, 2))
        if not is_error(r) and r > 1:
            assert sha256(dst[:r]) == z["out_sha256"][k]
            out = np.zeros(n + 2, np.uint8)
            if codec == 2:
                assert port.orc_fse_decompress_u16(ptr(out), n // 2, ptr(dst), r) == n // 2
            else:
                dr = (port.orc_fse_decompress if codec == 0 else port.orc_huf_decompress)(ptr(out), n, ptr(dst), r)
                if is_error(dr):
                    continue        # 1-bit code at tableLog 12: undecodable by the reference too (see test_oracle_vs_ref)
            assert np.array_equal(out[:n], d)
    assert {0, 1, 2} <= kinds
