"""Recorded calls into the compiled reference library, so that the tests comparing against it run without it.

The reference (the original C implementation, compiled by oracle/Makefile into oracle/_ref/libfse_ref.so) is not part
of this repository.  Every test that compares with it gets, from load_ref(), a stand-in that replays what the reference
returned and wrote in that test, recorded once where the reference was compiled (tests/golden/make_golden.py).

A call ref.NAME(*args) is served by a twin: the oracle port's equivalent of NAME, else (in the -m gpu suite) the product
library's function of that name, else nothing.  The recording holds, per call, the reference's return value, the bytes
where the reference left its buffer arguments different from the twin (as runs of bytes), and one byte of a digest
chained over all buffer arguments as the reference left them in this and every earlier call; the test's recording ends
with the whole 8-byte chain.  Replay runs the twin, writes those bytes, and checks the digest: the buffers the test
compares then hold exactly what the reference wrote, and a twin whose output changed since the recording fails the
check instead of standing in for the reference.  All tests' recordings are members of tests/golden/reference_calls.npz.

    FSE_RECORD_REFERENCE=DIR pytest tests ...     records with the compiled reference into DIR (one .npz per test)
    python tests/reference_calls.py DIR ...       merges such recordings into tests/golden/reference_calls.npz"""
import ctypes as C
import glob
import hashlib
import io
import os
import re
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_calls.npz")
RECORD_ENV = "FSE_RECORD_REFERENCE"

# buffer arguments the reference uses as scratch: neither recorded nor compared
SCRATCH_ARGS = {"HUF_compress4X_repeat": (6,), "HUF_compress1X_repeat": (6,)}

_current = None
_golden = None


def _dtable_is_x2(dt):
    return _buffer(dt)[1] != 0                               # DTableDesc {maxTableLog, tableType, tableLog, reserved}


PORT_TWINS = {"HIST_count": "orc_hist_count", "FSE_normalizeCount": "orc_fse_normalize", "FSE_NCountWriteBound": "orc_fse_ncount_bound",
              "FSE_writeNCount": "orc_fse_write_ncount", "FSE_readNCount": "orc_fse_read_ncount",
              "FSE_buildCTable": "orc_fse_build_ctable", "FSE_buildCTableU16": "orc_fse_build_ctable",
              "FSE_buildDTable": "orc_fse_build_dtable", "FSE_buildDTableU16": "orc_fse_build_dtable_u16",
              "FSE_compress_usingCTable": "orc_fse_encode", "FSE_decompress_usingDTable": "orc_fse_decode",
              "FSE_compress2": "orc_fse_compress2", "FSE_decompress": "orc_fse_decompress",
              "FSE_compressU16": "orc_fse_compress_u16", "FSE_decompressU16": "orc_fse_decompress_u16",
              "HUF_buildCTable": "orc_huf_build_ctable", "HUF_writeCTable": "orc_huf_write_ctable",
              "HUF_compress4X_usingCTable": "orc_huf_encode4x", "HUF_compress1X_usingCTable": "orc_huf_encode1x",
              "HUF_compress2": "orc_huf_compress2", "HUF_readStats": "orc_huf_read_stats",
              "HUF_readDTableX1": "orc_huf_read_dtable_x1", "HUF_readDTableX2": "orc_huf_read_dtable_x2",
              "HUF_decompress4X2_usingDTable": "orc_huf_decode4x2", "HUF_decompress1X2_usingDTable": "orc_huf_decode1x2",
              "HUF_decompress4X1_usingDTable": "orc_huf_decode4x1", "HUF_decompress1X1_usingDTable": "orc_huf_decode1x1",
              "HUF_decompress": "orc_huf_decompress", "HUF_decompress4X1": "orc_huf_decompress4x1",
              "HUF_decompress4X2": "orc_huf_decompress4x2", "HUF_selectDecoder": "orc_huf_select_decoder"}


def port_twins(P):
    """reference name -> the oracle port's function with the reference's arguments (pointers taken as void *)"""
    def loose(name):
        f0 = getattr(P, name); f = P[name]                   # P[name]: a function object of its own, for its own argtypes
        f.restype = f0.restype
        f.argtypes = [C.c_void_p if issubclass(t, C._Pointer) else t for t in f0.argtypes]
        return f
    t = {k: loose(v) for k, v in PORT_TWINS.items()}
    opt = loose("orc_optimal_tablelog")
    t["FSE_optimalTableLog"] = lambda tl, n, msv: opt(tl, n, msv, 2)
    t["HUF_optimalTableLog"] = lambda tl, n, msv: opt(tl, n, msv, 1)
    t["HUF_decompress4X_usingDTable"] = lambda d, n, s, k, dt: t["HUF_decompress4X" + "21"[not _dtable_is_x2(dt)] + "_usingDTable"](d, n, s, k, dt)
    t["HUF_decompress1X_usingDTable"] = lambda d, n, s, k, dt: t["HUF_decompress1X" + "21"[not _dtable_is_x2(dt)] + "_usingDTable"](d, n, s, k, dt)
    comp, decomp = loose("orc_compress_blocks"), loose("orc_decompress_blocks")
    t["refshim_compress_blocks"] = lambda *a: comp(*a[:-1])                 # last argument: the reference's thread count
    t["refshim_decompress_blocks"] = lambda *a: decomp(*a[:-1])
    return t


def _buffer(a):
    """writable byte view of the memory an argument points to, or None for a value argument"""
    if isinstance(a, C.c_void_p):
        if hasattr(a, "_arr"):                               # numpy's ndarray.ctypes.data_as keeps the array here
            arr = a._arr
            assert arr.flags.c_contiguous and arr.ctypes.data == a.value
            return arr.reshape(-1).view(np.uint8)
        assert not a.value, "a raw pointer argument: pass numpy arrays through helpers.ptr"
        return None
    if type(a).__name__ == "CArgObject":                     # ctypes.byref(x)
        a = a._obj
    if isinstance(a, (C.Array, C._SimpleCData)):
        return np.ctypeslib.as_array((C.c_uint8 * C.sizeof(a)).from_buffer(a))
    return None


def _chain(prev, bufs):
    h = hashlib.blake2b(prev, digest_size=8)
    for b in bufs:
        h.update(struct.pack("<q", -1 if b is None else len(b)))
        if b is not None:
            h.update(b)
    return h.digest()


def _encode_ret(r):
    if r is None:
        return 0, 3
    if isinstance(r, float):
        return struct.unpack("<Q", struct.pack("<d", r))[0], 2
    return r & (2 ** 64 - 1), (1 if r < 0 else 0)


def _decode_ret(v, kind):
    v = int(v)
    return [v, v - 2 ** 64, struct.unpack("<d", struct.pack("<Q", v))[0], None][kind]


def key_for(nodeid):
    mod, _, name = nodeid.partition("::")
    stem = os.path.splitext(os.path.basename(mod))[0] + "__" + name
    return re.sub(r"[^A-Za-z0-9_.-]", "_", stem.replace("[", "-").replace("]", ""))


def _runs(pos):
    """sorted positions -> (starts, lengths) of their runs of consecutive positions"""
    if not len(pos):
        return pos, pos
    cut = np.flatnonzero(np.diff(pos) != 1) + 1
    starts = pos[np.concatenate([[0], cut])]
    return starts, np.diff(np.concatenate([[0], cut, [len(pos)]]))


class _Fn:
    def __init__(self, lib, name):
        self.__dict__.update(_lib=lib, _name=name)

    def __setattr__(self, k, v):                            # restype / argtypes: for the reference and a product twin
        for f in (self._lib._real_fn(self._name), self._lib._product_fn(self._name)):
            if f is not None:
                setattr(f, k, v)

    def __call__(self, *args):
        return self._lib._call(self._name, args)


class RecordedReference:
    """load_ref()'s object for one test: records (FSE_RECORD_REFERENCE set, compiled reference present) or replays"""

    def __init__(self, nodeid, product=None):
        self.nodeid = nodeid
        self.key = key_for(nodeid)
        self.product = product
        self.product_fns = {}
        self.twins = None
        self.record_dir = os.environ.get(RECORD_ENV)
        self.real = None
        self.calls = []                                      # replay: the recording; record: what is being recorded
        self.pos = 0
        self.values = {}
        self.chain = b""
        self.final = b""
        if self.record_dir:
            from helpers import REF_SO
            assert os.path.exists(REF_SO), "recording needs the compiled reference " + REF_SO
            self.real = C.CDLL(REF_SO)
        else:
            self._load()

    # -- the library surface ----------------------------------------------------------------------------------------
    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        f = self.__dict__[name] = _Fn(self, name)            # one object per name: tests compare them with `is`
        return f

    def _real_fn(self, name):
        return getattr(self.real, name) if self.real is not None else None

    def _product_fn(self, name):
        """the product library's NAME as a function object of this recording's own (its argtypes leave the tests' alone)"""
        if self.product is None or name.startswith("refshim_"):
            return None
        if name not in self.product_fns:
            try:
                self.product_fns[name] = self.product[name]
            except AttributeError:
                self.product_fns[name] = None
        return self.product_fns[name]

    def _twin(self, name):
        """(function, what it is) computing NAME for the replay"""
        if self.twins is None:
            from helpers import load_port
            self.twins = port_twins(load_port())
        if name in self.twins:
            return self.twins[name], "the oracle port (oracle/fse_oracle.c)"
        f = self._product_fn(name)
        return (f, "the product library (libfse_b200.so)") if f is not None else (None, "nothing (the recording holds all of it)")

    def _call(self, name, args):
        skip = SCRATCH_ARGS.get(name, ())
        bufs = [None if i in skip else _buffer(a) for i, a in enumerate(args)]
        twin, twin_is = self._twin(name)
        if self.record_dir:
            pre = [None if b is None else b.copy() for b in bufs]
            if twin is not None:
                twin(*args)
            mine = [None if b is None else b.copy() for b in bufs]
            for b, p in zip(bufs, pre):
                if b is not None:
                    b[:] = p
            ret = getattr(self.real, name)(*args)
            diffs = []
            for i, (b, m) in enumerate(zip(bufs, mine)):
                if b is not None:
                    pos = np.flatnonzero(b != m)
                    for s, n in zip(*_runs(pos)):
                        diffs.append((i, int(s), b[s:s + n].copy()))
            self.chain = _chain(self.chain, bufs)
            self.calls.append((name, _encode_ret(ret), self.chain[0], diffs))
            return ret
        assert self.pos < len(self.calls), "%s: call %d (%s) is past the %d recorded reference calls%s" % (
            self.nodeid, self.pos, name, len(self.calls), "" if self.calls else " (no recording in " + GOLDEN + ")")
        rname, (rv, kind), digest, diffs = self.calls[self.pos]
        assert rname == name, "%s: call %d is %s, the recording has %s" % (self.nodeid, self.pos, name, rname)
        self.pos += 1
        if twin is not None:
            twin(*args)
        for i, s, val in diffs:
            bufs[i][s:s + len(val)] = val
        self.chain = _chain(self.chain, bufs)
        assert self.chain[0] == digest and (self.pos < len(self.calls) or self.chain == self.final), (
            "%s: call %d (%s) was computed by %s, and its result plus the recorded differences is no longer what the "
            "reference wrote: that code's output for this call changed since the recording, most likely a regression there "
            "(re-record only if the reference itself changed)" % (self.nodeid, self.pos - 1, name, twin_is))
        return _decode_ret(rv, kind)

    # -- small recorded facts (what a reference program printed or wrote, by digest) ---------------------------------
    def value(self, key, compute):
        if self.record_dir:
            self.values[key] = str(compute())
            return self.values[key]
        assert key in self.values, "%s: no recorded value %r in %s" % (self.nodeid, key, GOLDEN)
        return self.values[key]

    # -- storage: one npz per test while recording, one member per test in GOLDEN ------------------------------------
    def _load(self):
        global _golden
        if _golden is None:
            _golden = np.load(GOLDEN)
        if self.key not in _golden.files:
            return
        z = np.load(io.BytesIO(_golden[self.key].tobytes()))
        names = list(z["names"])
        ends = np.cumsum(z["d_len"])
        diffs = [[] for _ in range(len(z["fn"]))]
        for j, (k, i, s, n, e) in enumerate(zip(z["d_call"], z["d_arg"], z["d_start"], z["d_len"], ends)):
            diffs[k].append((int(i), int(s), z["d_val"][e - n:e]))
        self.calls = [(names[f], (r, k), dg, df) for f, r, k, dg, df in zip(z["fn"], z["ret"], z["ret_kind"], z["digest"], diffs)]
        self.final = z["final"].tobytes()
        self.values = dict(zip(z["value_keys"], z["values"]))

    def finish(self):
        if self.record_dir:
            if self.calls or self.values:
                self._save(os.path.join(self.record_dir, self.key + ".npz"))
            return
        assert self.pos == len(self.calls), "%s: %d of %d recorded reference calls made" % (self.nodeid, self.pos, len(self.calls))

    def _save(self, path):
        names = sorted({c[0] for c in self.calls})
        d = [(k, i, s, val) for k, c in enumerate(self.calls) for i, s, val in c[3]]
        np.savez(path, names=np.array(names if names else [""]), fn=np.array([names.index(c[0]) for c in self.calls], np.uint16),
                 ret=np.array([c[1][0] for c in self.calls], np.uint64), ret_kind=np.array([c[1][1] for c in self.calls], np.uint8),
                 digest=np.array([c[2] for c in self.calls], np.uint8), final=np.frombuffer(self.chain, np.uint8),
                 d_call=np.array([x[0] for x in d], np.uint32), d_arg=np.array([x[1] for x in d], np.uint8),
                 d_start=np.array([x[2] for x in d], np.uint32), d_len=np.array([len(x[3]) for x in d], np.int64),
                 d_val=np.concatenate([x[3] for x in d]) if d else np.zeros(0, np.uint8),
                 value_keys=np.array(list(self.values), dtype=str), values=np.array(list(self.values.values()), dtype=str))


def merge(dirs):
    """GOLDEN := its members, replaced or joined by the per-test recordings in `dirs`"""
    members = dict(np.load(GOLDEN)) if os.path.exists(GOLDEN) else {}
    for d in dirs:
        for f in sorted(glob.glob(os.path.join(d, "*.npz"))):
            members[os.path.basename(f)[:-4]] = np.fromfile(f, np.uint8)
    np.savez_compressed(GOLDEN, **dict(sorted(members.items())))


def begin(nodeid, product=None):
    global _current
    _current = RecordedReference(nodeid, product)


def end():
    global _current
    cur, _current = _current, None
    if cur is not None:
        cur.finish()


def active():
    return _current is not None


def current():
    assert _current is not None, "the recorded reference exists inside a test only"
    return _current


if __name__ == "__main__":
    import sys
    merge(sys.argv[1:])
