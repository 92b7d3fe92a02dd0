"""Helpers for the -m gpu suite: CPU-side compression with the checker (the reference: inside a test its recorded
calls, reference_calls.py; elsewhere, as in smoke(), the compiled library where it was built, else the oracle port)
into the bench.c slot layout."""
import ctypes as C
import os

import numpy as np

from helpers import load_port, load_ref, ptr

BLOCK = 32768
SLOT = 512 + BLOCK + (BLOCK >> 7) + 4 + 8
CODEC = {"fse": 0, "huf": 1, "u16": 2}


def checker():
    """(library, is_reference): the reference (inside a test its recorded calls, elsewhere the compiled library where
    oracle/_ref was built), else the oracle port"""
    ref = load_ref()
    if ref is not None:
        return ref, True
    return load_port(), False


def cpu_compress(codec, data, block=BLOCK, slot=None, msv=255, tl=12, threads=0):
    data = np.ascontiguousarray(data)
    slot = slot or (512 + block + (block >> 7) + 12)
    nb = (len(data) + block - 1) // block
    cbuf = np.zeros(nb * slot + 64, np.uint8)
    cs = np.zeros(nb, np.uint64)
    lib, isref = checker()
    if isref:
        lib.refshim_compress_blocks(CODEC[codec], ptr(data), len(data), block, ptr(cbuf), slot, ptr(cs), msv, tl,
                                    threads or (os.cpu_count() or 1))
    else:
        lib.orc_compress_blocks(CODEC[codec], ptr(data), len(data), block, ptr(cbuf), slot, ptr(cs), msv, tl)
    return cbuf, cs, slot


def cpu_decompress(codec, cbuf, cs, orig, block=BLOCK, slot=None, threads=0):
    orig = np.ascontiguousarray(orig)
    slot = slot or (512 + block + (block >> 7) + 12)
    nb = (len(orig) + block - 1) // block
    out = np.zeros(len(orig), np.uint8)
    res = np.zeros(nb, np.uint64)
    lib, isref = checker()
    if isref:
        lib.refshim_decompress_blocks(CODEC[codec], ptr(out), ptr(orig), len(orig), block, ptr(cbuf), slot, ptr(cs), ptr(res),
                                      threads or (os.cpu_count() or 1))
    else:
        lib.orc_decompress_blocks(CODEC[codec], ptr(out), ptr(orig), len(orig), block, ptr(cbuf), slot, ptr(cs), ptr(res))
    return out, res
