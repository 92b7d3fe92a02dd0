#!/usr/bin/env python
"""bench.py -- the judged benchmark: BASELINE.json's metric on BASELINE.json's config.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py ... --dump-outputs DIR      also writes the last timed step's outputs to DIR/*.npy (see dump_outputs)

Workload (config[1] of BASELINE.json): probagen P=14%, 1 GiB per GPU, Huff0 4X encode + decode on
32 KB blocks with the reference harness' parameters (maxSymbolValue 255, tableLog 12, slot =
FSE_compressBound(32768) = 33,548 B; programs/bench.c:98,113,355,569).  One STEP = HUF_compress2 of
every block of the batch followed by HUF_decompress of every block (one batched launch each).
  value  = uncompressed bytes that went through encode+decode per second, whole job (all GPUs),
           inputs resident in HBM, CUDA-event timed, max over ranks.
  e2e    = the same metric through the host-buffer C-ABI calls (FSEB200_compress_host /
           FSEB200_decompress_host): pinned host buffers, H2D/D2H copies inside the timed region.
  roofline = dominant kernel's algorithmic bytes (S read + C written for encode, C read + S written
           for decode; SURVEY.md 8d) / its CUDA-event duration, against MEASURED_PEAKS.json.
  cpu_baseline = the reference's own CPU path (oracle/_ref, compiled from the unmodified reference)
           on this box's host cores, same workload, timed in the same run (rank 0, N=1).
Multi-GPU: blocks are independent, so each rank owns a 1 GiB shard of the generator's stream
(weak scaling, no data-path collective); NCCL is only used for the barrier / max-over-ranks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 32768
SLOT = 512 + BLOCK + (BLOCK >> 7) + 4 + 8          # FSE_compressBound(32768), programs/bench.c:355
METRIC = "encode+decode GB/s (uncompressed) per GPU on 32 KB blocks; bit-exact vs ref"
CODEC_ID = {"fse": 0, "huf": 1, "u16": 2}


class Workload:
    """One BASELINE.json config: which codec, which generator, which call parameters.
      huf : configs[1]  probagen P=14%, HUF_compress2(.., 255, 12) / HUF_decompress, slot FSE_compressBound(32768)   (the headline)
      fse : configs[2]  probagen P=80%, FSE_compress2(.., 255, 12) / FSE_decompress
      u16 : configs[4]  generateU16(start 240, p 0.50, seed 1), 16384 symbols per block, FSE_compressU16(dst, 32768, .., 0, 12)
                        (programs/fuzzerU16.c:107-134, programs/bench.c:190-289, lib/fseU16.c:203-329)"""
    DEFAULT_P = {"huf": 0.14, "fse": 0.80, "u16": 0.50}

    def __init__(self, codec, p):
        self.codec = codec
        self.cid = CODEC_ID[codec]
        self.p = self.DEFAULT_P[codec] if p is None else p
        self.block = BLOCK
        self.slot = 32768 if codec == "u16" else SLOT
        self.msv, self.tl = (0, 12) if codec == "u16" else (255, 12)
        self.enc_kernels = {"huf": "huf_plan_kernel+huf_emit_kernel", "fse": "fse_encode_cta_kernel", "u16": "fse_encode_cta_kernel<U16>"}[codec]
        self.dec_kernels = {"huf": "huf_decode_kernel", "fse": "fse_decode_cta_kernel", "u16": "fse_decode_cta_kernel<U16>"}[codec]
        self.launches_per_step = {"huf": 5, "fse": 2, "u16": 2}[codec]   # huf: plan, emit, decode pass A, decode pass B (deferred list), x2 verdict sweep

    def describe(self, mib):
        if self.codec == "u16":
            return "generateU16 start=240 p=%.2f %d MiB per GPU (16384 16-bit symbols per 32 KB block), FSE-U16 encode+decode, FSE_compressU16(..,0,12)" % (self.p, mib)
        return "probagen P=%.0f%% %d MiB per GPU, %s encode+decode, 32 KB blocks, (255,12)" % (self.p * 100, mib, "Huff0 4X" if self.codec == "huf" else "FSE")

    def gen_device(self, L, ptr, nbytes, offset_bytes, stream):
        if self.codec == "u16":
            return L.FSEB200_genU16(ptr, nbytes // 2, offset_bytes // 2, 240, self.p, 1, stream)
        return L.FSEB200_probagen(ptr, nbytes, offset_bytes, self.p, stream)

    def gen_host(self, nbytes):
        import numpy as np
        port = os.path.join(ROOT, "oracle", "_build", "libfse_oracle.so")
        if not os.path.exists(port):
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
        L = C.CDLL(port)
        a = np.empty(nbytes, np.uint8)
        if self.codec == "u16":
            L.orc_gen_u16.restype = None
            L.orc_gen_u16.argtypes = [C.c_void_p, C.c_size_t, C.c_uint, C.c_double, C.c_uint32]
            L.orc_gen_u16(a.ctypes.data_as(C.c_void_p), nbytes // 2, 240, self.p, 1)
        else:
            L.orc_probagen.restype = None
            L.orc_probagen.argtypes = [C.c_void_p, C.c_size_t, C.c_double]
            L.orc_probagen(a.ctypes.data_as(C.c_void_p), nbytes, self.p)
        return a


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mib", type=int, default=1024, help="uncompressed MiB per GPU (BASELINE config: 1024)")
    ap.add_argument("--codec", default="huf", choices=["huf", "fse", "u16"], help="huf = BASELINE configs[1] (headline), fse = configs[2], u16 = configs[4]")
    ap.add_argument("--p", type=float, default=None, help="generator probability (default: the config's: huf 0.14, fse 0.80, u16 0.50)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sg", action="store_true", help="skip the separate scatter/decode/gather line at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (float32 / float64)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
# CPU checker access (bench.py is one of the few places allowed to execute oracle/)
# ------------------------------------------------------------------------------------------------
def load_checker():
    """(lib, kind): the compiled reference when its prebuilt .so travelled with the snapshot, else the port"""
    ref = os.path.join(ROOT, "oracle", "_ref", "libfse_ref.so")
    if os.path.exists(ref):
        L = C.CDLL(ref)
        L.refshim_compress_blocks.restype = C.c_double
        L.refshim_compress_blocks.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint, C.c_uint, C.c_int]
        L.refshim_decompress_blocks.restype = C.c_double
        L.refshim_decompress_blocks.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int]
        return L, "reference"
    port = os.path.join(ROOT, "oracle", "_build", "libfse_oracle.so")
    if not os.path.exists(port):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
    L = C.CDLL(port)
    L.orc_compress_blocks.restype = C.c_size_t
    L.orc_compress_blocks.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint, C.c_uint]
    L.orc_decompress_blocks.restype = C.c_size_t
    L.orc_decompress_blocks.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    return L, "port"


def cpu_roundtrip(L, kind, wl, data, cbuf, cs, out, res, threads):
    """one compress + decompress pass of the CPU implementation over `data`; returns (t_comp, t_decomp) seconds"""
    import numpy as np
    cid = wl.cid; SLOT = wl.slot
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    n = len(data)
    if kind == "reference":
        tc = L.refshim_compress_blocks(cid, p(data), n, BLOCK, p(cbuf), SLOT, p(cs), wl.msv, wl.tl, threads)
        td = L.refshim_decompress_blocks(cid, p(out), p(data), n, BLOCK, p(cbuf), SLOT, p(cs), p(res), threads)
        return tc, td
    nb = (n + BLOCK - 1) // BLOCK
    per = (nb + threads - 1) // threads

    def part(fn_c, t):
        b0 = t * per; b1 = min(nb, b0 + per)
        if b0 >= b1:
            return
        o = b0 * BLOCK; m = min(n, b1 * BLOCK) - o
        if fn_c:
            L.orc_compress_blocks(cid, data[o:].ctypes.data_as(C.c_void_p), m, BLOCK, cbuf[b0 * SLOT:].ctypes.data_as(C.c_void_p), SLOT,
                                  cs[b0:].ctypes.data_as(C.c_void_p), wl.msv, wl.tl)
        else:
            L.orc_decompress_blocks(cid, out[o:].ctypes.data_as(C.c_void_p), data[o:].ctypes.data_as(C.c_void_p), m, BLOCK,
                                    cbuf[b0 * SLOT:].ctypes.data_as(C.c_void_p), SLOT, cs[b0:].ctypes.data_as(C.c_void_p),
                                    res[b0:].ctypes.data_as(C.c_void_p))
    ts = []
    for fn_c in (True, False):
        th = [threading.Thread(target=part, args=(fn_c, t)) for t in range(threads)]
        t0 = time.perf_counter(); [x.start() for x in th]; [x.join() for x in th]; ts.append(time.perf_counter() - t0)
    return ts[0], ts[1]


def compare_all_blocks(codec, g_c, g_cs, w_c, w_cs, slot, nb):
    """every block: identical return value and identical compressed bytes.  Returns (ok, blocks compared, bytes compared, detail)."""
    import numpy as np
    g_cs = g_cs[:nb]; w_cs = w_cs[:nb]
    if not np.array_equal(g_cs, w_cs):
        bad = int(np.nonzero(g_cs != w_cs)[0][0])
        return False, nb, 0, "return value of block %d: %d vs reference %d" % (bad, int(g_cs[bad]), int(w_cs[bad]))
    sizes = w_cs.astype(np.int64).copy()
    sizes[w_cs > np.uint64(1 << 62)] = 0                      # in-band error codes store nothing
    if codec != "huf":
        sizes[sizes == 1] = 0                                  # FSE reports RLE as 1 and stores nothing; HUF stores the byte
    total = 0
    cols = np.arange(slot, dtype=np.int64)[None, :]
    for c0 in range(0, nb, 2048):
        k = min(2048, nb - c0)
        G = g_c[c0 * slot:(c0 + k) * slot].reshape(k, slot); W = w_c[c0 * slot:(c0 + k) * slot].reshape(k, slot)
        diff = (G != W) & (cols < sizes[c0:c0 + k, None])
        if diff.any():
            r, c = np.argwhere(diff)[0]
            return False, nb, total, "byte %d of block %d differs" % (int(c), c0 + int(r))
        total += int(sizes[c0:c0 + k].sum())
    return True, nb, total, None


DUMP_BLOCKS = 128                                  # blocks sampled by --dump-outputs over all ranks (see dump_outputs)


def dump_outputs(d, cbuf, cs, out, res, slot, rank=0, world=1):
    """What the encode and decode calls of the last timed step returned, as .npy files in `d`, so that two builds can be
    compared output for output: every block's encode return value (csizes) and decode return value (results) as float64
    (through int64, so an in-band error code 2^64 - k reads -k), and for a fixed, seeded sample of DUMP_BLOCKS // world
    blocks per rank (sample_blocks) their compressed bytes (the slot up to the block's return value, zeros after it) and
    decoded bytes as float32.  In all: DUMP_BLOCKS * (slot + 32 KB) * 4 B (34 MB) plus 16 B per block per rank (0.5 MB per
    GiB per rank), so at most 38 MB up to 8 ranks of 1 GiB.  With several ranks each writes <name>_rank<r>.npy.
    Takes numpy arrays or CUDA tensors."""
    import numpy as np

    def host(x):
        return x.cpu().numpy() if hasattr(x, "cpu") else x
    nb = len(cs)
    idx = np.sort(np.random.default_rng(1 + rank).choice(nb, min(nb, DUMP_BLOCKS // world), replace=False))
    sizes = host(cs).view(np.int64)
    comp = host(cbuf[:nb * slot].reshape(nb, slot)[idx]).astype(np.float32)
    used = np.where((sizes[idx] < 0) | (sizes[idx] > slot), 0, sizes[idx])                  # in-band error codes store nothing
    comp[np.arange(slot)[None, :] >= used[:, None]] = 0
    dec = host(out[:nb * BLOCK].reshape(nb, BLOCK)[idx]).astype(np.float32)
    suffix = "" if world == 1 else "_rank%d" % rank
    os.makedirs(d, exist_ok=True)
    for name, a in (("csizes", sizes.astype(np.float64)), ("results", host(res).view(np.int64).astype(np.float64)),
                    ("sample_blocks", idx.astype(np.float64)), ("compressed", comp), ("decoded", dec)):
        np.save(os.path.join(d, name + suffix + ".npy"), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's clocks line): one streaming
    `nvidia-smi -lms 20` process, every row time-stamped on arrival; summary() keeps the rows that fall inside
    [t0, t1] (the timed region) plus the closest neighbours when the region is shorter than the sampling period."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []; self.proc = None; self.index = index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [x.strip() for x in line.strip().split(",")]))
        except Exception:
            pass

    def start(self):
        self.t.start()
        t0 = time.perf_counter()                                   # nvidia-smi can take a second to print its first row on a cold box
        while len(self.rows) < 2 and time.perf_counter() - t0 < 5.0:
            time.sleep(0.05)

    def stop(self):
        time.sleep(0.05)
        if self.proc is not None:
            self.proc.terminate()
        self.t.join(timeout=3)

    def summary(self, t0, t1):
        inside = [r for (t, r) in self.rows if t0 <= t <= t1]
        if len(inside) < 3:                                        # very short region: take the nearest rows around it
            near = sorted(self.rows, key=lambda tr: abs(tr[0] - (t0 + t1) / 2))[:5]
            inside = [r for (_, r) in near]
        sm = sorted(int(float(r[0])) for r in inside if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in inside if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in inside if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in inside if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(inside), "samples_total": len(self.rows)}


def bind_to_gpu_numa_node(local):
    """Pin this rank (and, by first touch, the pinned host buffers it allocates next) to the NUMA node its GPU hangs off: on the
    8-GPU box GPUs 0-3 sit on node 0 and 4-7 on node 1, and a rank whose host buffers live on the other socket pays the
    inter-socket link on every PCIe transfer (round 1: e2e scaling efficiency 0.535 at N=8).  Best effort; returns what it did."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return {"numa_node": None, "note": "single-node host"}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        try:                                                       # memory policy: prefer the node (set_mempolicy, x86-64 syscall 238)
            libc = C.CDLL(None, use_errno=True)
            mask = C.c_ulong(1 << node)
            libc.syscall(238, 1, C.byref(mask), C.c_ulong(64))     # MPOL_PREFERRED
        except Exception:
            pass
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as exc:
        return {"numa_node": None, "note": repr(exc)[:80]}


def measured_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_note(kernel):
    """dram bytes per launch from the committed ncu capture of this same command (profiles/traffic.json names the capture it was
    read from), if one exists for this kernel: ncu cannot run inside the timed region, so this is a recorded measurement, not a
    live one -- the line says so in `traffic_source`."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t.get(kernel.split("(")[0])
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0                                                   # rank 0 alone times the CPU arm
    import numpy as np
    L, kind = load_checker()
    threads = os.cpu_count() or 1
    n = a.mib << 20
    if threads < 16:
        n = min(n, 256 << 20)                                     # bounded sample on small hosts
    wl = Workload(a.codec, a.p)
    SLOT = wl.slot
    data = wl.gen_host(n)
    nb = (n + BLOCK - 1) // BLOCK
    cbuf = np.zeros(nb * SLOT + 64, np.uint8); cs = np.zeros(nb, np.uint64)
    out = np.zeros(n, np.uint8); res = np.zeros(nb, np.uint64)
    for _ in range(max(a.warmup, 1)):
        cpu_roundtrip(L, kind, wl, data, cbuf, cs, out, res, threads)
    assert np.array_equal(out, data)
    tc = td = 0.0
    t0 = time.perf_counter()
    for _ in range(a.steps):
        x, y = cpu_roundtrip(L, kind, wl, data, cbuf, cs, out, res, threads); tc += x; td += y
    wall = time.perf_counter() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, cbuf, cs, out, res, SLOT)
    val = n * a.steps / (tc + td) / 1e9
    sample = "%d MiB of the workload's generator stream (%d blocks), all %d host threads, %d steps" % (n >> 20, nb, threads, a.steps)
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(1e3 * (tc + td) / a.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u16" if a.codec == "u16" else "u8", "data": "synthetic (restatement of the reference generator, seed 1)",
            "config": {"workload": wl.describe(n >> 20), "block_size": BLOCK, "slot": SLOT, "host_threads": threads},
            "encode_gbs": round(n * a.steps / tc / 1e9, 3), "decode_gbs": round(n * a.steps / td / 1e9, 3),
            "compressed_ratio": round(float(cs.astype(np.float64).sum()) / n, 5), "wall_s": round(wall, 2),
            "cpu_baseline": {"value": round(val, 3), "unit": "GB/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": round(val, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def run_b200(a):
    import numpy as np
    import torch
    import finitestateentropy_b200 as fb
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        # NCCL prints its version banner on stdout while the first communicator comes up: stdout must carry the JSON line only
        sys.stdout.flush(); saved_fd = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier(); torch.cuda.synchronize()
        finally:
            C.CDLL(None).fflush(None)                              # NCCL writes through libc's buffered stdout
            sys.stdout.flush(); os.dup2(saved_fd, 1); os.close(saved_fd)
    L = fb.lib()
    wl = Workload(a.codec, a.p)
    SLOT = wl.slot
    for nm, args in (("FSEB200_probagen", [C.c_void_p, C.c_size_t, C.c_size_t, C.c_double, C.c_void_p]),
                     ("FSEB200_genU16", [C.c_void_p, C.c_size_t, C.c_size_t, C.c_uint, C.c_double, C.c_uint, C.c_void_p]),
                     ("FSEB200_compress_host", [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_uint, C.c_uint]),
                     ("FSEB200_decompress_host", [C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p])):
        f = getattr(L, nm); f.restype = C.c_size_t; f.argtypes = args
    dev = torch.device("cuda", local)
    n = a.mib << 20
    nb = (n + BLOCK - 1) // BLOCK
    src = torch.empty(n, dtype=torch.uint8, device=dev)
    cbuf = torch.empty(nb * SLOT + 64, dtype=torch.uint8, device=dev)
    cs = torch.empty(nb, dtype=torch.int64, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    res = torch.empty(nb, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    assert wl.gen_device(L, src.data_ptr(), n, rank * n, stream) == 0            # this rank's shard of the generator stream
    enc = {"huf": fb.huf_compress_batch, "fse": fb.fse_compress_batch, "u16": fb.fseu16_compress_batch}[a.codec]
    dec = {"huf": fb.huf_decompress_batch, "fse": fb.fse_decompress_batch, "u16": fb.fseu16_decompress_batch}[a.codec]

    def step():
        enc(src, BLOCK, SLOT, wl.msv, wl.tl, cbuf=cbuf, csizes=cs)
        dec(cbuf, cs, n, BLOCK, SLOT, out=out, results=res, orig=src)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(a.warmup, 3)):
        step()
    torch.cuda.synchronize()
    # ---- parity gate of the run itself: round trip on every rank; on rank 0 EVERY block's return value and compressed bytes
    #      against the CPU checker's output for the same input (the whole shard where the host has the cores for it) ----
    ok_rt = bool(torch.equal(out, src)) and bool((res[:-1] == BLOCK).all())
    csum = int(cs.sum().item())
    bit_exact = None; bit_exact_detail = None; ref_pass = None
    if rank == 0:
        try:
            Lc, kind = load_checker()
            threads = os.cpu_count() or 1
            k = nb if threads >= 16 else min(nb, (256 << 20) // BLOCK)       # small hosts: bounded sample, said so in the line
            m = min(n, k * BLOCK)
            h = src[:m].cpu().numpy()
            wc = np.zeros(k * SLOT + 64, np.uint8); wcs = np.zeros(k, np.uint64); wo = np.zeros(m, np.uint8); wr = np.zeros(k, np.uint64)
            tc0, td0 = cpu_roundtrip(Lc, kind, wl, h, wc, wcs, wo, wr, threads)
            g_cs = cs[:k].cpu().numpy().view(np.uint64); g_c = cbuf[:k * SLOT].cpu().numpy()
            okb, nblk, nbytes, why = compare_all_blocks(a.codec, g_c, g_cs, wc, wcs, SLOT, k)
            # and the other direction: the GPU decodes the CHECKER's compressed blocks to the original bytes
            d_wc = torch.from_numpy(wc).to(dev); d_wcs = torch.from_numpy(wcs.view(np.int64)).to(dev)
            o2, r2 = dec(d_wc, d_wcs, m, BLOCK, SLOT, orig=src[:m])
            torch.cuda.synchronize()
            cross = bool(torch.equal(o2, src[:m]))
            del d_wc, d_wcs, o2, r2
            bit_exact = bool(okb and cross and np.array_equal(wo, h))
            bit_exact_detail = {"blocks_compared": nblk, "compressed_bytes_compared": nbytes, "of_blocks": nb, "checker": kind,
                                "gpu_decodes_checker_output": cross, "mismatch": why}
            ref_pass = (Lc, kind, h, wc, wcs, wo, wr, threads, m, k)
            del g_c
        except Exception as exc:                                   # checker unavailable: say so, do not guess
            bit_exact = "unchecked: %r" % (exc,)
    # ---- timed region: K steps, events on the launching (torch current) stream ----
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    wall0 = time.perf_counter()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(a.steps):
        ev[i][0].record(); enc(src, BLOCK, SLOT, wl.msv, wl.tl, cbuf=cbuf, csizes=cs)
        ev[i][1].record(); dec(cbuf, cs, n, BLOCK, SLOT, out=out, results=res, orig=src)
        ev[i][2].record()
    t1.record()
    barrier()
    wall1 = time.perf_counter()
    if sampler:
        sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, cbuf, cs, out, res, SLOT, rank, world)
    total_ms = t0.elapsed_time(t1)
    enc_ms = sum(ev[i][0].elapsed_time(ev[i][1]) for i in range(a.steps)) / a.steps
    dec_ms = sum(ev[i][1].elapsed_time(ev[i][2]) for i in range(a.steps)) / a.steps
    tm = torch.tensor([total_ms, enc_ms, dec_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms, enc_ms, dec_ms = [float(x) for x in tm.cpu()]
    value = world * n * a.steps / (total_ms * 1e-3) / 1e9

    # ---- end to end through the host-buffer C-ABI (pinned host memory, copies inside the timed region) ----
    e2e = None
    if not a.no_e2e:
        aff0 = os.sched_getaffinity(0)
        numa = bind_to_gpu_numa_node(local)
        h_src = torch.empty(n, dtype=torch.uint8, pin_memory=True); h_src.copy_(src)
        h_c = torch.empty(nb * SLOT + 64, dtype=torch.uint8, pin_memory=True)
        h_cs = torch.empty(nb, dtype=torch.int64, pin_memory=True)
        h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        h_res = torch.empty(nb, dtype=torch.int64, pin_memory=True)
        cid = wl.cid

        def host_step():
            r1 = L.FSEB200_compress_host(cid, h_c.data_ptr(), SLOT, h_cs.data_ptr(), h_src.data_ptr(), n, BLOCK, wl.msv, wl.tl)
            r2 = L.FSEB200_decompress_host(cid, h_out.data_ptr(), n, BLOCK, h_c.data_ptr(), SLOT, h_cs.data_ptr(), h_res.data_ptr(), h_src.data_ptr())
            assert r1 == 0 and r2 == 0
        host_step(); host_step()
        ok_e2e = bool(torch.equal(h_out, h_src))
        ke = max(1, min(a.steps, 3))
        barrier()
        w0 = time.perf_counter()
        for _ in range(ke):
            host_step()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        tw = torch.tensor([wall], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.cpu()[0])
        # bytes the two calls actually move (capi.cu: per 2048-block chunk the compressed side is copied as a strided 2-D
        # transfer of the widest block, rounded to 64 B; +16 B on the way in because the kernels read aligned 16-byte pieces)
        cs_np = h_cs.numpy()
        wid_out = wid_in = 0
        hchunk = int(os.environ.get("FSEB200_HOST_CHUNK_BLOCKS", "2048"))           # capi.cu chunk_blocks()
        for c0 in range(0, nb, hchunk):
            mx = int(cs_np[c0:c0 + hchunk].max()); cbk = min(hchunk, nb - c0)
            wid_out += min(SLOT, (mx + 63) & ~63) * cbk
            wid_in += min(SLOT, (mx + 16 + 63) & ~63) * cbk
        e2e = {"value": round(world * n * ke / wall / 1e9, 3), "unit": "GB/s", "steps": ke, "roundtrip_ok": ok_e2e,
               "h2d_bytes_per_step": n + wid_in + 8 * nb, "d2h_bytes_per_step": wid_out + 8 * nb + n + 8 * nb,
               "host_binding": numa,
               "api": "FSEB200_compress_host + FSEB200_decompress_host (pinned host buffers, %d-block chunks on 4 streams)" % hchunk,
               "note": "PCIe-bound: each of the two calls moves the uncompressed GiB one way (19.3 ms at the measured 55.6 GB/s) while the "
                       "compressed side goes the other way; both one-way bounds together cap this metric at about 28 GB/s per GPU"}
        del h_src, h_c, h_out
        try:                                                       # the CPU baseline below must see every core again
            os.sched_setaffinity(0, aff0)
            C.CDLL(None).syscall(238, 0, None, C.c_ulong(0))       # MPOL_DEFAULT
        except Exception:
            pass

    # ---- BASELINE configs[3] shape, reported separately (SURVEY 8e): the root scatters the compressed shards over NVLink, every
    #      rank decodes its shard, the root gathers the decoded shards.  Bounded by the root's NVLink port, not by the codec:
    #      (N-1) GiB must come back through it (about 770 GB/s measured per direction).  So the work is cut to fit the link:
    #        * only USED bytes travel: each shard is re-pitched on the root from 33,548-byte slots to rows of the widest block
    #          (+ slack for the decoder's 32-byte reads); the decoder takes any slot stride, so nobody unpacks anything;
    #        * the shard is cut into K pieces, and scatter (root egress) and gather (root ingress) use two NCCL communicators,
    #          i.e. two streams: piece k+1 goes out while piece k is decoded and piece k-1 comes back. ----
    sg = None
    if dist is not None and world > 1 and not a.no_sg and a.codec == "huf":
        # pieces: a decode launch lasts one "round" -- about 0.5 ms for a piece of <= 512 MiB (the decoder packs small batches into few
        # CTAs), 0.95 ms for a GiB -- so cut no finer than what keeps a piece's decode under the time the root needs to take the
        # previous piece back, (N-1) * piece / 770 GB/s:  K <= 2.8 (N-1), i.e. 2 pieces at N=2, 8 at N=4 and N=8.
        K = 1
        while K < 8 and 2 * K <= 2.8 * (world - 1) and nb % (2 * K) == 0:
            K *= 2
        nbk = nb // K                                               # blocks per piece
        wmax = cs.max().reshape(1).clone()
        dist.all_reduce(wmax, op=dist.ReduceOp.MAX)                 # one pitch for every shard
        W = (int(wmax.item()) + 32 + 63) // 64 * 64                 # widest block + the decoder's 32-byte read-ahead, 64-byte multiple
        W = min(W, SLOT)
        pg_s = dist.new_group(list(range(world))); pg_g = dist.new_group(list(range(world)))
        packed = cbuf[:nb * SLOT].view(nb, SLOT)[:, :W].contiguous()                    # [nb, W] (setup, on every rank)
        pad = torch.zeros(64, dtype=torch.uint8, device=dev)
        root_c = root_s = parts_o = None
        if rank == 0:
            root_c = [torch.empty(nb * W + 64, dtype=torch.uint8, device=dev) for _ in range(world)]
            root_s = [torch.empty_like(cs) for _ in range(world)]
            parts_o = [torch.empty_like(out) for _ in range(world)]
        mine_c = torch.cat([packed.view(-1), pad])
        dist.gather(mine_c, root_c, dst=0); dist.gather(cs, root_s, dst=0)             # setup: the root now holds every shard, packed
        rc = torch.empty(nb * W + 64, dtype=torch.uint8, device=dev); rs = torch.empty_like(cs)
        cur = torch.cuda.current_stream()

        def piece_c(t, k):
            return t[k * nbk * W: (k + 1) * nbk * W + (64 if k == K - 1 else 0)]

        def sg_step():
            if rank == 0:
                works = []
                for k in range(K):                                   # egress: piece k of every shard, one NCCL group per piece
                    ops = [dist.P2POp(dist.isend, piece_c(root_c[r], k), r, pg_s) for r in range(1, world)]
                    ops += [dist.P2POp(dist.isend, root_s[r][k * nbk:(k + 1) * nbk], r, pg_s) for r in range(1, world)]
                    works += dist.batch_isend_irecv(ops)
                for k in range(K):                                   # ingress: decoded piece k of every shard
                    ops = [dist.P2POp(dist.irecv, parts_o[r][k * nbk * BLOCK:(k + 1) * nbk * BLOCK], r, pg_g) for r in range(1, world)]
                    works += dist.batch_isend_irecv(ops)
                for k in range(K):                                   # the root's own shard, piece by piece like everybody else
                    dec(piece_c(root_c[0], k), root_s[0][k * nbk:(k + 1) * nbk], nbk * BLOCK, BLOCK, W,
                        out=parts_o[0][k * nbk * BLOCK:(k + 1) * nbk * BLOCK], results=res[k * nbk:(k + 1) * nbk], orig=None)
                for w in works:
                    w.wait()
            else:
                recvs = []
                for k in range(K):
                    recvs.append(dist.batch_isend_irecv([dist.P2POp(dist.irecv, piece_c(rc, k), 0, pg_s),
                                                         dist.P2POp(dist.irecv, rs[k * nbk:(k + 1) * nbk], 0, pg_s)]))
                sends = []
                for k in range(K):
                    for w in recvs[k]:
                        w.wait()                                     # the compute stream waits for piece k (no host block)
                    dec(piece_c(rc, k), rs[k * nbk:(k + 1) * nbk], nbk * BLOCK, BLOCK, W,
                        out=out[k * nbk * BLOCK:(k + 1) * nbk * BLOCK], results=res[k * nbk:(k + 1) * nbk], orig=None)
                    sends += dist.batch_isend_irecv([dist.P2POp(dist.isend, out[k * nbk * BLOCK:(k + 1) * nbk * BLOCK], 0, pg_g)])
                for w in sends:
                    w.wait()
        out.zero_()
        sg_step()
        barrier()
        g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True)
        ks = 3
        g0.record()
        for _ in range(ks):
            sg_step()
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        okt = torch.tensor([1 if torch.equal(out if rank else parts_o[0], src) else 0], dtype=torch.int32, device=dev)
        if rank == 0:                                               # every gathered shard is the generator's stream for that rank
            chk = torch.empty_like(src)
            for r in range(1, world):
                assert wl.gen_device(L, chk.data_ptr(), n, r * n, stream) == 0
                okt &= int(torch.equal(parts_o[r], chk))
            del chk
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        ok_sg = bool(int(okt.cpu()[0]))
        ms = float(tg.cpu()[0]) / ks
        link = 770.0                                                # GB/s per direction per GPU, measured (B200_PROFILING.md)
        bound_ms = max((world - 1) * n, (world - 1) * nb * W) / link / 1e6
        sg = {"what": "BASELINE configs[3]: root scatters compressed Huff0 shards (rows re-pitched to the widest block, %d pieces), all ranks "
                      "decode, root gathers decoded shards; scatter and gather on separate NCCL communicators so egress / decode / ingress overlap" % K,
              "decode_gbs_incl_transfers": round(world * n / (ms * 1e-3) / 1e9, 2), "ms_per_step": round(ms, 3), "steps": ks,
              "bytes_scattered": (world - 1) * nb * W, "bytes_gathered": (world - 1) * n, "row_pitch": W, "pieces": K,
              "root_link_bound_ms": round(bound_ms, 3), "frac_of_link_bound": round(bound_ms / ms, 3), "roundtrip_ok": ok_sg}
        del root_c, parts_o, rc, packed, mine_c

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    # ---- roofline of the dominant kernel (algorithmic bytes: S + C each way, SURVEY.md 8d) ----
    peak, peak_src = measured_peak()
    alg = n + csum
    kern = {wl.enc_kernels: enc_ms, wl.dec_kernels: dec_ms}
    dom = max(kern, key=kern.get)
    roof = lambda ms: round(alg / (ms * 1e-3) / 1e9, 2)
    roofline = {"kernel": dom, "bound": "hbm", "achieved": roof(kern[dom]), "peak": peak, "unit": "GB/s",
                "frac": round(roof(kern[dom]) / peak, 4), "traffic": traffic_note(dom),
                "traffic_source": "profiles/traffic.json: ncu --set full capture of this command (dram__bytes_read.sum + dram__bytes_write.sum per launch), round 2" if traffic_note(dom) else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg,
                "all_kernels": {k: {"ms": round(v, 4), "achieved": roof(v), "frac": round(roof(v) / peak, 4)} for k, v in kern.items()}}
    # ---- the reference's CPU path on this box's host cores, same run (N=1 only) ----
    cpu = None
    if world == 1 and not a.no_cpu:
        try:
            if ref_pass is None:
                raise RuntimeError("checker unavailable")
            Lc, kind, h, wc, wcs, wo, wr, threads, m, k = ref_pass
            reps = 3; tc = td = 0.0
            for _ in range(reps):
                x, y = cpu_roundtrip(Lc, kind, wl, h, wc, wcs, wo, wr, threads); tc += x; td += y
            one = min(m, 64 << 20)
            x1, y1 = cpu_roundtrip(Lc, kind, wl, h[:one], wc, wcs, wo, wr, 1)
            cpu = {"value": round(m * reps / (tc + td) / 1e9, 3), "unit": "GB/s", "cores": threads, "kind": kind,
                   "sample": "%d MiB of the same input, %d reps, encode %.2f GB/s + decode %.2f GB/s" % (m >> 20, reps, m * reps / tc / 1e9, m * reps / td / 1e9),
                   "single_thread": {"value": round(one / (x1 + y1) / 1e9, 4), "encode_gbs": round(one / x1 / 1e9, 4), "decode_gbs": round(one / y1 / 1e9, 4),
                                     "sample": "%d MiB" % (one >> 20)}}
        except Exception as exc:
            cpu = {"value": None, "unit": "GB/s", "cores": 0, "kind": "unavailable", "sample": repr(exc)}
    line = {"metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": round(total_ms / a.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u16" if a.codec == "u16" else "u8", "data": "synthetic (reference generator restated, generated in HBM, seed 1, shard = rank * size)",
            "config": {"workload": wl.describe(a.mib), "block_size": BLOCK, "slot": SLOT, "blocks_per_gpu": nb, "l2": "inputs (%d MiB) larger than the 126 MB L2" % a.mib,
                       "sharding": "independent blocks, contiguous shard per rank, no data-path collective"},
            "encode_gbs_per_gpu": round(n / (enc_ms * 1e-3) / 1e9, 2), "decode_gbs_per_gpu": round(n / (dec_ms * 1e-3) / 1e9, 2),
            "per_gpu": round(value / world, 3), "compressed_ratio": round(csum / n, 5),
            "bit_exact": bit_exact, "bit_exact_detail": bit_exact_detail, "roundtrip_ok": ok_rt,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "scatter_gather": sg, "gpu_launches": wl.launches_per_step * a.steps,
            "clocks": sampler.summary(wall0, wall1) if sampler else None}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    args = parse()
    sys.exit(run_reference(args) if args.impl == "reference" else run_b200(args))
