#!/usr/bin/env python3
"""bench.py -- the contract benchmark of the batched-decompress hot path.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--codec snappy|lz4|cascaded|bitcomp|ans]

One "step" = one pass of the hot path over one batch of 10,000 x 64 KB synthetic chunks per GPU through the C ABI
of libnvcomp.so (nvcompBatched<Fmt>DecompressAsync).  Default workload = BASELINE.json configs[1]: Snappy batched
decompress, 10,000 x 64 KB synthetic tabular float32 chunks, 1 GPU.  The metric is the reference's: total
uncompressed bytes / (1e9 * seconds), CUDA-event timed around the asynchronous call (reference
benchmarks/benchmark_template_chunked.cuh:519-539,604-607).

Prints ONE JSON line (rank 0):
  value          N = 1: device-resident decode throughput.  N > 1: the whole job north_star describes -- rank 0 owns the
                 compressed slab of every rank's chunk range, scatters it over NCCL (NVLink) in slices on a side stream
                 while the slices already received are decoded; `decode_only` stands beside it
  e2e            the same decode with HOST buffers (pinned): H2D + decode + D2H inside the timed region
  roofline       algorithmic bytes / event-timed launch duration vs the measured HBM peak
  per_dataset    the survey's own cfg2 definitions: (i) reference gen_data(3), (ii) price-walk float32 column
  foreign_streams  the same workload compressed on the HOST by an independent codec (pyarrow-snappy / liblz4 default
                 and HC-12) and decoded on the GPU, parity-gated
  cfg1           (--codec lz4) BASELINE configs[0]: 16 x 64 KB LZ4 round trip, latency in us next to liblz4 on one core
  cpu_baseline   liblz4's LZ4_decompress_safe (LZ4) / the oracle port on this box's host cores, median and best
  cfg5           (N > 1, or --cfg5) BASELINE configs[4]: LZ4, 80,000 x 64 KB chunks in total, strong scaling
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK = 65536
CHUNKS_PER_GPU = 10000
CFG5_TOTAL_CHUNKS = 80000
FMT = {"lz4": "LZ4", "snappy": "Snappy", "cascaded": "Cascaded", "bitcomp": "Bitcomp", "ans": "ANS"}
ORACLE_ID = {"lz4": 0, "snappy": 1, "cascaded": 2, "bitcomp": 3, "ans": 4, "liblz4": 5}
DEFAULT_DATASET = {"lz4": "lz4_mixed", "snappy": "tabular_f32", "cascaded": "sorted_i64",
                   "bitcomp": "sorted_i64", "ans": "lowentropy_bytes"}
KERNEL_NAME = {"lz4": "lz4_decompress_v2_kernel (+ lz4_decompress_light_kernel beside it)",
               "snappy": "snappy_decompress_v2_kernel (+ snappy_decompress_light_kernel beside it)",
               "cascaded": "cascaded_decompress_kernel", "bitcomp": "bitcomp_decompress_kernel",
               "ans": "ans_decompress_kernel"}
WORKLOAD_NAME = {
    "snappy": "BASELINE configs[1]: Snappy batched decompress, 10000x64KB synthetic tabular float32 chunks per GPU",
    "lz4": "BASELINE configs[4] per-GPU share: LZ4 batched decompress, 10000x64KB chunks (run-length int32 + tabular float32) per GPU",
    "cascaded": "BASELINE configs[2]: Cascaded (RLE+delta+bitpack) decompress, sorted int64, 10000x64KB per GPU",
    "bitcomp": "Bitcomp decompress, sorted int64, 10000x64KB per GPU",
    "ans": "BASELINE configs[3]: ANS batched decompress, 10000x64KB low-entropy byte chunks per GPU",
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def codec_opts(kind: str, dataset: str):
    from nvcomp_b200._lib import BitcompOpts, CascadedOpts, Type
    if kind == "cascaded":
        return CascadedOpts(4096, Type.LONGLONG if "i64" in dataset else Type.INT, 1, 1, 1)
    if kind == "bitcomp":
        return BitcompOpts(0, Type.ULONGLONG if "i64" in dataset else Type.UINT)
    return None


# ----------------------------------------------------------------------------------------------
# host placement: pin the rank to the NUMA node of its GPU before any pinned allocation
# ----------------------------------------------------------------------------------------------
def pin_to_gpu_numa(gpu_index: int) -> dict:
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return {"pinned": False, "why": "no pci bus id"}
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return {"pinned": False, "why": "numa_node = -1 (single node or not exposed)"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"pinned": True, "numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001 -- placement is best effort, the numbers say whether it mattered
        return {"pinned": False, "why": f"{type(e).__name__}: {e}"}


# ----------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------
# CPU codecs (baseline legs only): the oracle port and liblz4 through oracle/batch.c's pthread runner
# ----------------------------------------------------------------------------------------------
def load_oracle():
    path = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", ROOT, "oracle/liboracle.so"], check=True, stdout=subprocess.DEVNULL)
    lib = C.CDLL(path)
    lib.oracle_batch_decompress.restype = C.c_double
    lib.oracle_batch_decompress.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                            C.c_size_t, C.c_void_p, C.c_int]
    lib.oracle_have_liblz4.restype = C.c_int
    return lib


def cpu_decode_time(lib, codec_id, comp_host, offs, lens, out_host, threads) -> float:
    out_len = np.zeros(len(offs), dtype=np.uint64)
    t = lib.oracle_batch_decompress(codec_id, comp_host.ctypes.data, offs.ctypes.data, lens.ctypes.data,
                                    len(offs), out_host.ctypes.data, CHUNK, out_len.ctypes.data, threads)
    if t < 0 or not (out_len == CHUNK).all():
        raise RuntimeError("CPU decoder failed on the sample")
    return t


def cpu_time_stats(lib, codec_id, comp_host, offs, lens, raw_check, threads, steps=None, budget_s=4.0):
    """The one estimator both the cpu_baseline leg and --impl reference use: wall time of every repetition
    (oracle/batch.c: last worker finish - first worker start), reported as median and best."""
    n = len(offs)
    out_host = np.empty(n * CHUNK, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    lens = np.ascontiguousarray(lens, dtype=np.uint64)
    cpu_decode_time(lib, codec_id, comp_host, offs, lens, out_host, threads)      # warm-up + correctness
    if raw_check is not None and not np.array_equal(out_host[: raw_check.size], raw_check.reshape(-1)):
        raise RuntimeError("CPU decoder output differs from the original data")
    times, t_start = [], time.time()
    while (len(times) < steps) if steps else (len(times) < 3 or (time.time() - t_start < budget_s and len(times) < 200)):
        times.append(cpu_decode_time(lib, codec_id, comp_host, offs, lens, out_host, threads))
    return {"median_GBps": n * CHUNK / float(np.median(times)) / 1e9, "best_GBps": n * CHUNK / min(times) / 1e9,
            "reps": len(times), "median_s": float(np.median(times))}


def cpu_baseline(kind, comp_host, offs, lens, raw_check):
    lib = load_oracle()
    threads = os.cpu_count() or 1
    n = len(offs)
    port = cpu_time_stats(lib, ORACLE_ID[kind], comp_host, offs, lens, raw_check, threads)
    out = {"value": round(port["median_GBps"], 2), "unit": "GB/s", "cores": threads, "kind": "port",
           "estimator": "median of the repetitions (best beside it); the same estimator as --impl reference",
           "best_GBps": round(port["best_GBps"], 2),
           "sample": f"{n} chunks x 64 KB of this workload (the GPU-compressed streams), {port['reps']} repetitions, "
                     f"oracle/ C decoder, {threads} pthreads (contiguous chunk range per thread)"}
    if kind == "lz4" and lib.oracle_have_liblz4():
        ref = cpu_time_stats(lib, ORACLE_ID["liblz4"], comp_host, offs, lens, raw_check, threads)
        out.update({"value": round(ref["median_GBps"], 2), "best_GBps": round(ref["best_GBps"], 2), "kind": "reference",
                    "port_median_GBps": round(port["median_GBps"], 2), "port_best_GBps": round(port["best_GBps"], 2),
                    "sample": f"{n} chunks x 64 KB of this workload, {ref['reps']} repetitions, liblz4.so.1 "
                              f"LZ4_decompress_safe (the CPU decoder the reference links, examples/lz4_cpu_decompression.cu:"
                              f"143-147; dlopen), {threads} pthreads; the oracle port is reported beside it"})
    return out


# ----------------------------------------------------------------------------------------------
# workload construction
# ----------------------------------------------------------------------------------------------
def gen_data(dataset: str, n_chunks: int, seed_offset: int = 0):
    from nvcomp_b200 import datagen
    if ":" in dataset:
        name, col = dataset.split(":")
        return datagen.tabular_f32(n_chunks, column=int(col), **({"seed": 1000 * seed_offset + 1} if seed_offset else {}))
    gen = datagen.DATASETS[dataset]
    try:
        return gen(n_chunks, seed=1000 * seed_offset + gen.__defaults__[0]) if seed_offset else gen(n_chunks)
    except TypeError:
        return gen(n_chunks)


def device_batch(data: np.ndarray):
    import torch
    from nvcomp_b200.batched import Batch
    n = data.shape[0]
    slab = torch.from_numpy(data.reshape(-1)).cuda()
    offsets = np.arange(n, dtype=np.int64) * CHUNK
    return Batch(slab, torch.from_numpy(offsets + slab.data_ptr()).cuda(),
                 torch.full((n,), CHUNK, dtype=torch.int64, device="cuda"), offsets)


def compact(comp, align=16):
    """Pack the compressed chunks contiguously (what a file / network sender would hold)."""
    import torch
    sizes = comp.sizes.cpu().numpy().astype(np.int64)
    al = (sizes + align - 1) // align * align
    offs = np.concatenate([[0], np.cumsum(al)[:-1]]).astype(np.int64)
    total = int(al.sum())
    dense = torch.zeros(total + 64, dtype=torch.uint8, device="cuda")
    for i in range(len(sizes)):
        o, src_o, sz = int(offs[i]), int(comp.offsets[i]), int(sizes[i])
        dense[o: o + sz] = comp.slab[src_o: src_o + sz]
    return dense, offs, sizes


def host_slab_to_batch(chunks):
    """list of bytes -> (dense device slab, offsets, sizes) in the same 16-byte aligned packing as compact()."""
    import torch
    sizes = np.array([len(c) for c in chunks], dtype=np.int64)
    al = (sizes + 15) // 16 * 16
    offs = np.concatenate([[0], np.cumsum(al)[:-1]]).astype(np.int64)
    host = np.zeros(int(al.sum()) + 64, dtype=np.uint8)
    for c, o in zip(chunks, offs):
        host[o:o + len(c)] = np.frombuffer(c, dtype=np.uint8)
    return torch.from_numpy(host).cuda(), offs, sizes


class Workload:
    """One compressed batch resident in HBM + everything a decode launch needs."""

    def __init__(self, kind, dataset, n, seed_offset=0, data=None, comp_chunks=None):
        import torch
        from nvcomp_b200.batched import Batch, Codec, empty_batch
        self.kind, self.dataset, self.n = kind, dataset, n
        self.data = gen_data(dataset, n, seed_offset) if data is None else data
        self.inp = device_batch(self.data)
        self.codec = Codec(FMT[kind], opts=codec_opts(kind, dataset))
        if comp_chunks is None:
            strided = self.codec.compress(self.inp, max_chunk=CHUNK)
            torch.cuda.synchronize()
            self.dense, self.c_offs, self.c_sizes = compact(strided)
            del strided
        else:
            self.dense, self.c_offs, self.c_sizes = host_slab_to_batch(comp_chunks)
        dev = self.dense.device
        self.comp = Batch(self.dense, torch.from_numpy(self.c_offs + self.dense.data_ptr()).cuda(),
                          torch.from_numpy(self.c_sizes).cuda(), self.c_offs)
        self.comp_total = int(self.c_sizes.sum())
        self.comp_span = int(self.c_offs[-1] + self.c_sizes[-1])
        self.total = n * CHUNK
        self.out = empty_batch(n, CHUNK)
        self.tb = self.codec.decompress_get_temp_size(n, CHUNK)
        self.temp = torch.empty(max(self.tb, 1), dtype=torch.uint8, device=dev)
        self.actual = torch.zeros(n, dtype=torch.int64, device=dev)
        self.status = torch.full((n,), -1, dtype=torch.int32, device=dev)

    def launch(self, stream_handle, ptrs=None, a=0, b=None, temp=None):
        b = self.n if b is None else b
        ptrs = self.comp.ptrs if ptrs is None else ptrs
        temp = self.temp if temp is None else temp
        self.codec.decompress_async(ptrs.data_ptr() + 8 * a, self.comp.sizes.data_ptr() + 8 * a,
                                    self.inp.sizes.data_ptr() + 8 * a, self.actual.data_ptr() + 8 * a, b - a,
                                    temp.data_ptr(), self.tb, self.out.ptrs.data_ptr() + 8 * a,
                                    self.status.data_ptr() + 4 * a, stream_handle)

    def check(self):
        import torch
        torch.cuda.synchronize()
        if not (bool((self.status == 0).all().item()) and bool((self.actual == CHUNK).all().item())):
            st, ac = self.status.cpu().numpy(), self.actual.cpu().numpy()
            bad = np.nonzero((st != 0) | (ac != CHUNK))[0]
            raise AssertionError(f"decompress status/size: {len(bad)} of {self.n} chunks, first {bad[:8].tolist()}, "
                                 f"status {st[bad[:8]].tolist()}, actual {ac[bad[:8]].tolist()}, "
                                 f"comp sizes {self.c_sizes[bad[:8]].tolist()}")
        assert torch.equal(self.out.slab[: self.total], self.inp.slab[: self.total]), "decompressed bytes differ from the input"

    def reset_outputs(self):
        self.out.slab.zero_(); self.status.fill_(-1); self.actual.zero_()

    def alg_bytes(self):
        return self.total + self.comp_total + 44 * self.n


def time_decode(w: Workload, steps: int, warmup: int):
    """CUDA events on the launching stream around every launch and around the whole timed region."""
    import torch
    sh = torch.cuda.current_stream().cuda_stream
    for _ in range(max(warmup, 3)):
        w.launch(sh)
    w.check()                       # parity gate before timing: bit-exact vs the original data, every status success
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for a, b in evs:
        a.record()
        w.launch(sh)
        b.record()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, [a.elapsed_time(b) for a, b in evs]


DUMP_SAMPLE_CHUNKS = 200     # 200 x 64 KB as float32 = 52 MB, inside the 64 MB a dump may take


def dump_outputs(w: Workload, out_dir: str):
    """What a caller of nvcompBatched<Fmt>DecompressAsync received in the last timed step, as .npy (float32 /
    float64) so two builds can be compared output for output: every chunk's status and decompressed size, and the
    decompressed bytes of a fixed, seeded sample of the chunks (all of them when the batch is small enough)."""
    import torch
    torch.cuda.synchronize()
    k = min(w.n, DUMP_SAMPLE_CHUNKS)
    idx = np.sort(np.random.default_rng(0).choice(w.n, size=k, replace=False))
    slab = w.out.slab[: w.n * CHUNK].view(w.n, CHUNK)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"statuses": w.status.cpu().numpy().astype(np.float32),
              "decompressed_sizes": w.actual.cpu().numpy().astype(np.float64),
              "sample_chunk_index": idx.astype(np.float64),
              "sample_chunks": slab[torch.from_numpy(idx).to(slab.device)].cpu().numpy().astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def rate_line(w: Workload, ms: float, peak: float):
    return {"chunks": w.n, "ratio": round(w.total / w.comp_total, 3), "GBps": round(w.total / ms / 1e6, 1),
            "ms": round(ms, 4), "roofline_frac": round(w.alg_bytes() / ms / 1e6 / peak, 4)}


# ----------------------------------------------------------------------------------------------
# the multi-GPU job: rank 0 owns every rank's compressed slab and scatters it while the ranks decode
# ----------------------------------------------------------------------------------------------
class DistributedJob:
    NSLICES = 4

    def __init__(self, w: Workload, rank: int, world: int):
        import torch
        import torch.distributed as dist
        self.w, self.rank, self.world = w, rank, world
        dev = w.dense.device
        n = w.n
        self.bounds = [n * i // self.NSLICES for i in range(self.NSLICES + 1)]
        self.spans = [(int(w.c_offs[a]), int(w.c_offs[b - 1] + w.c_sizes[b - 1])) for a, b in zip(self.bounds, self.bounds[1:])]
        # setup (untimed): rank 0 collects every rank's compressed slab + slice table -- "rank 0 owns the input"
        meta = torch.tensor([w.comp_span] + [x for s in self.spans for x in s], dtype=torch.int64, device=dev)
        metas = [torch.zeros_like(meta) for _ in range(world)]
        dist.all_gather(metas, meta)
        self.metas = [m.cpu().tolist() for m in metas]
        self.owned = {}
        if rank == 0:
            for r in range(1, world):
                self.owned[r] = torch.empty(self.metas[r][0], dtype=torch.uint8, device=dev)
                dist.recv(self.owned[r], r)
        else:
            dist.send(w.dense[: w.comp_span].contiguous(), 0)
            self.recv_buf = torch.zeros(w.comp_span + 64, dtype=torch.uint8, device=dev)
            self.recv_ptrs = torch.from_numpy(w.c_offs + self.recv_buf.data_ptr()).to(dev)
        self.comm = torch.cuda.Stream()
        self.dstreams = [torch.cuda.Stream() for _ in range(self.NSLICES)]
        self.temps = [torch.empty(max(w.tb, 1), dtype=torch.uint8, device=dev) for _ in range(self.NSLICES)]
        self.dist = dist
        self.torch = torch

    def step(self, decode=True):
        """One job: every slice of every remote rank's share leaves rank 0 on the comm stream; a rank decodes slice i
        on its own stream as soon as it has arrived (one 2,500-chunk launch alone would be bounded by the latency of a
        single chunk, so the slices' launches overlap); rank 0 decodes its own share from the slab it already holds."""
        torch, dist, w = self.torch, self.dist, self.w
        cur = torch.cuda.current_stream()
        self.comm.wait_stream(cur)                       # the previous job's decode has consumed the buffers
        works = []
        with torch.cuda.stream(self.comm):
            for i in range(self.NSLICES):
                if self.rank == 0:
                    ops = []
                    for r in range(1, self.world):
                        lo, hi = self.metas[r][1 + 2 * i], self.metas[r][2 + 2 * i]
                        ops.append(dist.P2POp(dist.isend, self.owned[r][lo:hi], r))
                    works.append(dist.batch_isend_irecv(ops) if ops else [])
                else:
                    lo, hi = self.spans[i]
                    works.append(dist.batch_isend_irecv([dist.P2POp(dist.irecv, self.recv_buf[lo:hi], 0)]))
        if decode and self.rank == 0:
            w.launch(cur.cuda_stream)                    # own share: nothing to wait for, one launch
        elif decode:
            for i in range(self.NSLICES):
                a, b = self.bounds[i], self.bounds[i + 1]
                st = self.dstreams[i]
                st.wait_stream(cur)
                with torch.cuda.stream(st):
                    for wk in works[i]:
                        wk.wait()                        # this slice's stream waits for this slice only
                    w.launch(st.cuda_stream, ptrs=self.recv_ptrs, a=a, b=b, temp=self.temps[i])
            for st in self.dstreams:
                cur.wait_stream(st)
        else:
            for ws in works:
                for wk in ws:
                    wk.wait()
        if self.rank == 0 and decode:
            for ws in works:
                for wk in ws:
                    wk.wait()

    def timed(self, steps, warmup, decode=True):
        torch, dist = self.torch, self.dist
        for _ in range(max(warmup, 3)):
            self.step(decode)
        torch.cuda.synchronize()
        if decode:
            self.w.check()
            if self.rank != 0:
                assert torch.equal(self.recv_buf[: self.w.comp_span], self.w.dense[: self.w.comp_span]), "scattered slab differs"
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step(decode)
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=self.w.dense.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


def measure(kind, dataset, n, rank, world, args, sampler=None):
    """Decode-only timing (every N) and, for N > 1, the distribution-inclusive job."""
    import torch
    import torch.distributed as dist
    w = Workload(kind, dataset, n, seed_offset=rank)
    dev = w.dense.device
    if sampler is not None:
        sampler.start()
    if world > 1:
        dist.barrier()
    ms_dec, launch_ms = time_decode(w, args.steps, args.warmup)
    res = {"w": w, "launch_ms": launch_ms}
    if world > 1:
        t = torch.tensor([ms_dec], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dec = float(t.item())
        cs = torch.tensor([float(w.comp_total)], device=dev)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
        res["comp_total_all"] = float(cs.item())
        w.reset_outputs()
        job = DistributedJob(w, rank, world)
        ms_job = job.timed(args.steps, args.warmup, decode=True)
        ms_comm = job.timed(max(3, args.steps // 2), 3, decode=False)
        sent = res["comp_total_all"] - w.comp_total if rank == 0 else 0.0
        st = torch.tensor([sent], device=dev)
        dist.all_reduce(st, op=dist.ReduceOp.MAX)
        res.update({"ms_job": ms_job, "ms_comm": ms_comm, "bytes_sent_by_rank0": float(st.item())})
    else:
        res["comp_total_all"] = float(w.comp_total)
    res["ms_dec"] = ms_dec
    return res


def cfg1_latency():
    """BASELINE configs[0] (reference benchmark_lz4_synth.cpp:64-72): LZ4 round trip of 1 MB of synthetic int32
    run-length data as 16 x 64 KB chunks on one GPU -- a latency figure (one launch over 16 chunks is far from filling
    the GPU), next to liblz4 on one host core over the same chunks."""
    import torch
    n = 16
    w = Workload("lz4", "runlength_i32", n)
    sh = torch.cuda.current_stream().cuda_stream
    codec = w.codec
    ctb = codec.compress_get_temp_size(n, CHUNK)
    ctemp = torch.empty(max(ctb, 1), dtype=torch.uint8, device=w.dense.device)
    from nvcomp_b200.batched import empty_batch
    max_out = codec.compress_get_max_output_chunk_size(CHUNK)
    cout = empty_batch(n, max_out)
    csz = torch.zeros(n, dtype=torch.int64, device=w.dense.device)

    def timed(fn, reps=60, warm=5):
        for _ in range(warm):
            fn()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        t = sorted(a.elapsed_time(b) * 1e3 for a, b in evs)
        return t[len(t) // 2], t[0]

    c_med, c_best = timed(lambda: codec.compress_async(w.inp.ptrs.data_ptr(), w.inp.sizes.data_ptr(), CHUNK, n,
                                                       ctemp.data_ptr(), ctb, cout.ptrs.data_ptr(), csz.data_ptr(), sh))
    d_med, d_best = timed(lambda: w.launch(sh))
    w.check()
    out = {"workload": "BASELINE configs[0]: LZ4 round trip, 16 x 64 KB int32 run-length chunks (1 MB), one launch each way",
           "ratio": round(w.total / w.comp_total, 2),
           "gpu_compress_us": round(c_med, 1), "gpu_decompress_us": round(d_med, 1),
           "gpu_decompress_best_us": round(d_best, 1),
           "gpu_decompress_GBps": round(w.total / d_med / 1e3, 2),
           "what": "CUDA events around one CompressAsync / DecompressAsync over the 16 chunks, median of 60 (device-resident)"}
    try:
        lz4 = C.CDLL("liblz4.so.1")
        lz4.LZ4_compress_default.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int]
        lz4.LZ4_decompress_safe.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int]
        cap = CHUNK + CHUNK // 255 + 64
        raws = [w.data[i].tobytes() for i in range(n)]
        bufs = [C.create_string_buffer(cap) for _ in range(n)]
        outb = C.create_string_buffer(CHUNK)
        ct, dt = [], []
        for _ in range(20):
            t0 = time.perf_counter()
            sizes = [lz4.LZ4_compress_default(r, b, CHUNK, cap) for r, b in zip(raws, bufs)]
            t1 = time.perf_counter()
            for b, sz in zip(bufs, sizes):
                lz4.LZ4_decompress_safe(b, outb, sz, CHUNK)
            t2 = time.perf_counter()
            ct.append((t1 - t0) * 1e6); dt.append((t2 - t1) * 1e6)
        out.update({"liblz4_compress_us": round(sorted(ct)[10], 1), "liblz4_decompress_us": round(sorted(dt)[10], 1),
                    "liblz4": "liblz4.so.1 LZ4_compress_default / LZ4_decompress_safe, one host thread, the 16 chunks in turn "
                              "(includes the ctypes call overhead, ~1 us per chunk), median of 20"})
    except OSError:
        out["liblz4"] = "liblz4.so.1 not found on this box"
    return out


def foreign_streams(kind, base: Workload, args, peak):
    """The same chunks compressed on the HOST by an independent codec, decoded on the GPU (bit-exact gate)."""
    from concurrent.futures import ThreadPoolExecutor
    out = {}
    producers = []
    n = base.n
    if kind == "snappy":
        import pyarrow as pa
        codec = pa.Codec("snappy")
        producers.append(("pyarrow_snappy", n, lambda raw: codec.compress(raw).to_pybytes()))
    elif kind == "lz4":
        lz4 = C.CDLL("liblz4.so.1")
        lz4.LZ4_compress_default.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int]
        lz4.LZ4_compress_HC.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int]
        cap = CHUNK + CHUNK // 255 + 64

        def lz4_default(raw):
            buf = C.create_string_buffer(cap)
            n_ = lz4.LZ4_compress_default(raw, buf, len(raw), cap)   # before buf.raw: that makes a copy
            return buf.raw[:n_]

        def lz4_hc(raw):
            buf = C.create_string_buffer(cap)
            n_ = lz4.LZ4_compress_HC(raw, buf, len(raw), cap, 12)
            return buf.raw[:n_]
        producers.append(("liblz4_default", n, lz4_default))
        producers.append(("liblz4_hc12", min(n, 4000), lz4_hc))     # HC-12 is slow to produce: bounded sample, stated
    for name, m, fn in producers:
        data = base.data[:m]
        with ThreadPoolExecutor(max_workers=min(64, os.cpu_count() or 1)) as ex:
            chunks = list(ex.map(lambda i: fn(data[i].tobytes()), range(m)))
        # a sample smaller than the batch is decoded reps times over (every stream into its own output chunk), so
        # the launch fills the GPU like the other lines: a 4000-chunk launch is one partial wave of warps
        reps = max(1, -(-n // m))
        if reps > 1:
            data, chunks = np.concatenate([data] * reps), chunks * reps
        w = Workload(kind, base.dataset, m * reps, data=data, comp_chunks=chunks)
        ms, _ = time_decode(w, max(5, args.steps // 2), 3)
        out[name] = rate_line(w, ms, peak)
        if reps > 1:
            out[name]["distinct_chunks"] = m
        del w
    return out


# ----------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa = pin_to_gpu_numa(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)

    kind = args.codec
    dataset = args.dataset or DEFAULT_DATASET[kind]
    n = args.chunks
    peak, peak_src = peaks()
    sampler = ClockSampler(torch.cuda.current_device()) if rank == 0 else None
    m = measure(kind, dataset, n, rank, world, args, sampler)
    w = m["w"]
    if rank == 0 and args.dump_outputs:
        dump_outputs(w, args.dump_outputs)
    if rank == 0:
        # the timed region lasts only tens of ms; keep the identical load running (untimed) until the
        # sampler has seen ~0.6 s of it, so the clock record describes this kernel under load
        sh = torch.cuda.current_stream().cuda_stream
        t_load = time.time()
        while time.time() - t_load < 0.6:
            for _ in range(10):
                w.launch(sh)
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + 0.6 s of the same launches (untimed), nvidia-smi -lms 20"

    # ---- e2e: host buffers in, host buffers out, through the same C-ABI call, pipelined in slices
    e2e = run_e2e(w, args, world)
    e2e_dev = run_e2e(w, args, world, copy_back=False)

    total = w.total
    ms_dec = m["ms_dec"]
    decode_only = world * total / (ms_dec * 1e-3) / 1e9
    if world > 1:
        ms_per_step = m["ms_job"]
        value = world * total / (ms_per_step * 1e-3) / 1e9
    else:
        ms_per_step, value = ms_dec, decode_only
    avg_launch_ms = float(np.mean(m["launch_ms"]))
    alg_bytes = w.alg_bytes()
    achieved = alg_bytes / (avg_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        traffic = tj.get(f"{kind}:{dataset}")
        traffic_src = tj.get("_source", "profiles/traffic.json")

    line = {
        "metric": "decompressed GB/s (64KB chunks), whole job",
        "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME[kind], "codec": kind, "dataset": dataset, "chunks_per_gpu": n,
                   "chunk_bytes": CHUNK, "compression_ratio": round(world * total / m["comp_total_all"], 3),
                   "l2_policy": "inputs larger than L2 (compressed + decompressed footprint per step = "
                                f"{(total + w.comp_total) / 1e6:.0f} MB vs 126 MB L2)",
                   "sharding": ("contiguous chunk range per rank; rank 0 owns the compressed slab of every range and scatters "
                                f"it over NCCL in {DistributedJob.NSLICES} slices per rank, overlapped with the decode of the "
                                "slices that have arrived (inside `value`)") if world > 1 else "single GPU",
                   "host_placement": numa},
        "decode_only": {"value": round(decode_only, 2), "unit": "GB/s", "ms_per_step": round(ms_dec, 4),
                        "what": "the decode launches alone, inputs resident (no distribution), max over ranks"},
        "e2e": e2e,
        "e2e_device_consumer": e2e_dev,
        # kernels of this library inside the timed region, per rank: an LZ DecompressAsync is three launches
        # (classification, dense decoder, light decoder), the others one; the N > 1 job decodes in NSLICES calls per
        # step (rank 0: one call on the slab it holds)
        "gpu_launches": (3 if kind in ("lz4", "snappy") else 1) * args.steps * (DistributedJob.NSLICES if world > 1 else 1),
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic,
                     "traffic_source": traffic_src or "not captured for this workload",
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                     "kernel": KERNEL_NAME[kind], "avg_launch_ms": round(avg_launch_ms, 4)},
        "clocks": clocks,
    }
    if world > 1:
        line["distribute"] = {
            "what": "the job's NCCL scatter alone (no decode), warm, max over ranks: bytes leaving rank 0 per step / time",
            "bytes": int(m["bytes_sent_by_rank0"]), "ms": round(m["ms_comm"], 3),
            "GBps": round(m["bytes_sent_by_rank0"] / (m["ms_comm"] * 1e-3) / 1e9, 1)}

    if rank == 0 and world == 1:
        if kind in ("lz4", "snappy") and not args.no_extras:
            per = {}
            for name, ds in (("cfg2_i_gen_data3", "snappy_synth"), ("cfg2_ii_price_walk_f32", "tabular_f32:0")):
                wd = Workload(kind, ds, n)
                ms, _ = time_decode(wd, max(5, args.steps // 2), 3)
                per[name] = rate_line(wd, ms, peak)
                del wd
            line["per_dataset"] = per
            line["foreign_streams"] = foreign_streams(kind, w, args, peak)
            if kind == "lz4":
                line["cfg1"] = cfg1_latency()
        if not args.no_cpu:
            sample = min(n, args.cpu_chunks)
            host = w.dense[: int(w.c_offs[sample - 1] + w.c_sizes[sample - 1])].cpu().numpy()
            line["cpu_baseline"] = cpu_baseline(kind, host, w.c_offs[:sample], w.c_sizes[:sample], w.data[:sample])

    # ---- BASELINE configs[4]: LZ4, 80,000 x 64 KB in total, strong scaling (N > 1 always; N = 1 with --cfg5)
    if world > 1 or args.cfg5:
        m.clear()
        del w
        torch.cuda.empty_cache()
        n5 = CFG5_TOTAL_CHUNKS // world
        m5 = measure("lz4", "lz4_mixed", n5, rank, world, args)
        t5 = world * n5 * CHUNK
        cfg5 = {"workload": "BASELINE configs[4]: LZ4 batched decompress, 80000x64KB chunks (run-length int32 + tabular "
                            "float32) sharded by contiguous chunk range", "scaling": "strong", "chunks_total": world * n5,
                "chunks_per_gpu": n5,
                "decode_only": {"GBps": round(t5 / (m5["ms_dec"] * 1e-3) / 1e9, 2), "ms": round(m5["ms_dec"], 4)}}
        if world > 1:
            cfg5["job"] = {"GBps": round(t5 / (m5["ms_job"] * 1e-3) / 1e9, 2), "ms": round(m5["ms_job"], 4),
                           "what": "rank 0 scatters every other rank's share over NCCL, overlapped with decode"}
            cfg5["distribute"] = {"bytes": int(m5["bytes_sent_by_rank0"]), "ms": round(m5["ms_comm"], 3),
                                  "GBps": round(m5["bytes_sent_by_rank0"] / (m5["ms_comm"] * 1e-3) / 1e9, 1)}
        line["cfg5"] = cfg5
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(w: Workload, args, world, copy_back=True):
    """Same decode through the C ABI, but the compressed chunks start in pinned HOST memory and the
    decompressed chunks end in pinned HOST memory; both copies are inside the timed region.  The batch is
    processed in slices, one stream per slice (H2D -> decode -> D2H in order on it), so the copies of one
    slice overlap the decode of another and both copy engines stay busy."""
    import torch
    import torch.distributed as dist
    from nvcomp_b200.batched import empty_batch
    dev = w.dense.device
    n, total, comp_total = w.n, w.total, w.comp_span
    c_offs, c_sizes = w.c_offs, w.c_sizes
    h_comp = torch.empty(comp_total, dtype=torch.uint8).pin_memory()
    h_comp.copy_(w.dense[:comp_total])
    h_out = torch.empty(total, dtype=torch.uint8).pin_memory()
    d_comp = torch.empty(comp_total + 64, dtype=torch.uint8, device=dev)
    out = empty_batch(n, CHUNK)
    ptrs = torch.from_numpy(c_offs + d_comp.data_ptr()).to(dev)
    sizes = torch.from_numpy(c_sizes).to(dev)
    caps = w.inp.sizes
    actual = torch.zeros(n, dtype=torch.int64, device=dev)
    status = torch.full((n,), -1, dtype=torch.int32, device=dev)
    h_status = torch.empty(n, dtype=torch.int32).pin_memory()
    nslices = 8
    bounds = [n * i // nslices for i in range(nslices + 1)]
    streams = [torch.cuda.Stream() for _ in range(nslices)]
    tb = w.tb
    temps = [torch.empty(max(tb, 1), dtype=torch.uint8, device=dev) for _ in range(nslices)]
    codec = w.codec

    def step():
        for i in range(nslices):
            a, b = bounds[i], bounds[i + 1]
            lo, hi = int(c_offs[a]), int(c_offs[b - 1] + c_sizes[b - 1])
            st = streams[i]
            with torch.cuda.stream(st):
                d_comp[lo:hi].copy_(h_comp[lo:hi], non_blocking=True)
                codec.decompress_async(ptrs.data_ptr() + 8 * a, sizes.data_ptr() + 8 * a, caps.data_ptr() + 8 * a,
                                       actual.data_ptr() + 8 * a, b - a, temps[i].data_ptr(), tb,
                                       out.ptrs.data_ptr() + 8 * a, status.data_ptr() + 4 * a, st.cuda_stream)
                if copy_back:
                    h_out[a * CHUNK: b * CHUNK].copy_(out.slab[a * CHUNK: b * CHUNK], non_blocking=True)
                h_status[a:b].copy_(status[a:b], non_blocking=True)

    def drain():
        for st in streams:
            st.synchronize()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ok = bool((h_status == 0).all().item()) and (not copy_back or np.array_equal(
        h_out.numpy()[: 4 * CHUNK], w.inp.slab[: 4 * CHUNK].cpu().numpy()))
    assert ok, "e2e output mismatch"
    if world > 1:
        dist.barrier()
    steps = max(3, min(args.steps, 10))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
        drain()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if not copy_back:
        return {"value": round(world * total / (ms * 1e-3) / 1e9, 2), "unit": "GB/s",
                "h2d_bytes_per_step": comp_total, "d2h_bytes_per_step": 4 * n, "ms_per_step": round(ms, 3),
                "what": "same call, decompressed chunks stay in HBM for a GPU consumer; only statuses return"}
    return {"value": round(world * total / (ms * 1e-3) / 1e9, 2), "unit": "GB/s",
            "h2d_bytes_per_step": comp_total, "d2h_bytes_per_step": total + 4 * n,
            "ms_per_step": round(ms, 3), "pipeline": f"{nslices} slices, one stream each (H2D -> decode -> D2H)",
            "what": "pinned host compressed chunks -> H2D -> nvcompBatched*DecompressAsync -> D2H of the "
                    "decompressed chunks and statuses into pinned host memory (PCIe-bound: "
                    "d2h_bytes/ms_per_step is the link rate)"}


def oracle_compress_batch(lib, kind, dataset, data: np.ndarray):
    """Compress every chunk with the CPU oracle's own encoders (reference arm: no CUDA code of this repo runs)."""
    from concurrent.futures import ThreadPoolExecutor
    u8p, sz = C.c_char_p, C.c_size_t
    n = data.shape[0]
    cap = 2 * CHUNK + 65536
    t64 = "i64" in dataset
    if kind in ("lz4", "snappy", "ans"):
        fn = getattr(lib, f"oracle_{kind}_compress")
        fn.argtypes, fn.restype = [u8p, sz, u8p, sz], C.c_long
        call = lambda raw, out: fn(raw, len(raw), out, cap)
    elif kind == "cascaded":
        fn = lib.oracle_cascaded_compress
        fn.argtypes, fn.restype = [u8p, sz, u8p, sz, sz, C.c_uint, C.c_int, C.c_int, C.c_int], C.c_long
        call = lambda raw, out: fn(raw, len(raw), out, cap, 4096, 6 if t64 else 4, 1, 1, 1)
    else:
        fn = lib.oracle_bitcomp_compress
        fn.argtypes, fn.restype = [u8p, sz, u8p, sz, C.c_uint, C.c_uint], C.c_long
        call = lambda raw, out: fn(raw, len(raw), out, cap, 0, 7 if t64 else 5)

    def one(i):
        out = C.create_string_buffer(cap)
        r = call(data[i].tobytes(), out)
        assert r > 0
        return out.raw[:r]

    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        comps = list(ex.map(one, range(n)))
    sizes = np.array([len(c) for c in comps], dtype=np.int64)
    al = (sizes + 15) // 16 * 16
    offs = np.concatenate([[0], np.cumsum(al)[:-1]]).astype(np.int64)
    slab = np.zeros(int(al.sum()) + 64, dtype=np.uint8)
    for c, o in zip(comps, offs):
        slab[o:o + len(c)] = np.frombuffer(c, dtype=np.uint8)
    return slab, offs, sizes


def run_reference(args):
    """--impl reference: the reference's own implementation of this path is the closed libnvcomp.so
    (not in /root/reference, not installable: no source, no wheel).  Per the task's tier rules this arm
    times the CPU implementation of the path instead, on all host cores, on the same workload: for LZ4 the decoder
    the reference itself links for its known-answer tests (liblz4's LZ4_decompress_safe, dlopen'd), for the other
    codecs the oracle port (oracle/*.c).  Nothing of libnvcomp.so is loaded on this arm: the synthetic chunks are
    compressed by the oracle's own CPU encoders."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    kind = args.codec
    dataset = args.dataset or DEFAULT_DATASET[kind]
    n = min(args.chunks, args.cpu_chunks)
    data = gen_data(dataset, n)
    lib = load_oracle()
    host, c_offs, c_sizes = oracle_compress_batch(lib, kind, dataset, data)
    threads = os.cpu_count() or 1
    use_liblz4 = kind == "lz4" and bool(lib.oracle_have_liblz4())
    st = cpu_time_stats(lib, ORACLE_ID["liblz4"] if use_liblz4 else ORACLE_ID[kind], host, c_offs, c_sizes, data, threads,
                        steps=max(args.steps, 3))
    v = st["median_GBps"]
    decoder = ("liblz4.so.1 LZ4_decompress_safe (dlopen)" if use_liblz4 else "oracle/ C decoder")
    sample = (f"{n} chunks x 64 KB per step ({'same batch size' if n == args.chunks else 'bounded sample'} as the GPU arm's "
              f"workload, same generator), oracle/ C encoders, {decoder}, {threads} pthreads, median of {st['reps']} steps")
    line = {
        "impl": "reference", "metric": "decompressed GB/s (64KB chunks), whole job", "value": round(v, 2),
        "unit": "GB/s", "n_gpus": world, "steps": st["reps"], "warmup": 1,
        "ms_per_step": round(st["median_s"] * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME[kind], "codec": kind, "dataset": dataset, "chunks_per_gpu": n,
                   "chunk_bytes": CHUNK, "compression_ratio": round(n * CHUNK / float(c_sizes.sum()), 3),
                   "note": "the reference library is closed-source and absent; CPU implementation of the path "
                           "on the host cores, per the task's reference-arm rule"},
        "cpu_baseline": {"value": round(v, 2), "unit": "GB/s", "cores": threads, "kind": "reference" if use_liblz4 else "port",
                         "sample": sample, "best_GBps": round(st["best_GBps"], 2),
                         "estimator": "median of the steps (best beside it); the same estimator as the GPU arm's cpu_baseline"},
        "e2e": {"value": round(v, 2), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--codec", default="snappy", choices=sorted(FMT))
    ap.add_argument("--dataset", default=None)
    ap.add_argument("--chunks", type=int, default=CHUNKS_PER_GPU)
    ap.add_argument("--cpu-chunks", type=int, default=10000, help="bounded CPU sample (chunks)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip per_dataset / foreign_streams (kernel iteration)")
    ap.add_argument("--cfg5", action="store_true", help="also run BASELINE configs[4] (80,000 LZ4 chunks) at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step decompressed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
