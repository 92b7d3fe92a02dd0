"""SURVEY.md section 8f-2: the `.fse` frame format (programs/fileio.c:266-626) through programs/fse_b200_file.c.

The reference's own command-line tool (`fse`, compiled from the unmodified sources by oracle/Makefile `cli` into
oracle/_ref/fse_ref) is the checker: a frame written by our tool must be BYTE-IDENTICAL to the one `fse -e` / `fse -h`
writes for the same input, and each tool must decode the other's output -- the `make check` round trip of
programs/Makefile:115-131, plus raw / RLE / partial blocks and every block-size id.  What the reference tool wrote and
decoded is replayed as SHA-256 digests recorded with it (reference_calls.py)."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from helpers import load_ref, probagen

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OURS = os.path.join(ROOT, "programs", "_bin", "fse_b200_file")
REF = os.path.join(ROOT, "oracle", "_ref", "fse_ref")


def _run(args):
    r = subprocess.run(args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (args, r.stdout[-500:], r.stderr[-800:])


def _sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def _ref_output(args, out):
    """digest of the file the reference tool writes to `out` (while recording)"""
    _run([REF, "-f"] + [str(x) for x in args] + [str(out)])
    return _sha(out)


def _inputs():
    rng = np.random.default_rng(21)
    yield "proba20", probagen(1048575, 0.20)                       # `make check`'s input (programs/Makefile:117)
    yield "proba80", probagen(300000, 0.80)
    mixed = np.concatenate([probagen(32768 * 3, 0.14), rng.integers(0, 256, 32768 * 2, dtype=np.uint8),      # raw blocks
                            np.full(32768 * 2 + 777, 7, np.uint8), probagen(5000, 0.3)])                     # RLE blocks + a partial tail
    yield "mixed", mixed
    yield "tiny", np.arange(11, dtype=np.uint8)
    yield "exact", probagen(32768 * 4, 0.14)                       # multiple of the block size: no trailing empty block


@pytest.mark.parametrize("flag", ["-e", "-h"])
def test_frames_are_byte_identical_to_the_reference_tool_and_cross_decode(tmp_path, flag):
    if not os.path.exists(OURS):
        pytest.skip("fse_b200_file not built")
    ref = load_ref()
    for name, data in _inputs():
        src = tmp_path / (name + ".bin"); data.tofile(src)
        a = tmp_path / (name + ".ours.fse"); b = tmp_path / (name + ".ref.fse")
        _run([OURS, flag, str(src), str(a)])
        want = ref.value("%s %s frame" % (name, flag), lambda: _ref_output([flag, src], b))
        assert _sha(a) == want, (name, flag)
        da = tmp_path / (name + ".ours.out"); db = tmp_path / (name + ".ref.out")
        _run([OURS, "-d", str(a), str(da)])                        # we decode the reference's frame (identical to ours)
        theirs = ref.value("%s %s decoded" % (name, flag), lambda: _ref_output(["-d", a], db))      # the reference decodes ours
        assert open(da, "rb").read() == data.tobytes() and theirs == hashlib.sha256(data.tobytes()).hexdigest(), (name, flag)


def test_empty_input_round_trips(tmp_path):
    """an empty file is a header + trailer frame (the reference tool itself dies on it: integer division by zero in its
    statistics line, fileio.c:425 -- so there is nothing to compare against, only our own round trip)"""
    if not os.path.exists(OURS):
        pytest.skip("fse_b200_file not built")
    src = tmp_path / "e.bin"; open(src, "wb").close()
    for flag in ("-e", "-h"):
        _run([OURS, flag, str(src), str(tmp_path / "e.fse")])
        assert os.path.getsize(tmp_path / "e.fse") == 8
        _run([OURS, "-d", str(tmp_path / "e.fse"), str(tmp_path / "e.out")])
        assert os.path.getsize(tmp_path / "e.out") == 0


def test_every_block_size_id_and_corruption_is_detected(tmp_path):
    if not os.path.exists(OURS):
        pytest.skip("fse_b200_file not built")
    ref = load_ref()
    data = probagen(200000, 0.14)
    src = tmp_path / "in.bin"; data.tofile(src)
    for bid in range(0, 7):
        a = tmp_path / ("b%d.fse" % bid); o = tmp_path / ("b%d.out" % bid)
        _run([OURS, "-h", "-B%d" % bid, str(src), str(a)])
        # the frame the reference decoded when this was recorded, and what it decoded it to
        theirs = ref.value("-B%d frame decoded" % bid, lambda: _sha(a) + " " + _ref_output(["-d", a], o))
        assert theirs == _sha(a) + " " + hashlib.sha256(data.tobytes()).hexdigest(), bid
        _run([OURS, "-d", str(a), str(o)])
        assert open(o, "rb").read() == data.tobytes()
    frame = bytearray(open(tmp_path / "b5.fse", "rb").read())
    frame[len(frame) // 2] ^= 0x10
    bad = tmp_path / "bad.fse"; open(bad, "wb").write(frame)
    r = subprocess.run([OURS, "-d", str(bad), str(tmp_path / "bad.out")], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0                                       # decoding error or checksum mismatch, as the reference reports
