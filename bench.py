#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the seekstorm_b200 hot path.

Metric (BASELINE.json): queries/sec at top-10.  N=1 workload = configs[1]: brute-force cosine kNN over
1M x 768 f32 (C2).  A "step" = one call of the hot path over one batch of synthetic queries (batch = --batch
queries = batch/16 corpus passes).  `value` = device-resident QPS (queries already in HBM, packed keys left
in HBM); `e2e` = the same through the reference-facing C-ABI call ssb_search_vector with HOST buffers (H2D of
the queries and D2H of the results inside the timed region).  A second section ("bm25") measures C3
(BM25 OR top-10 over a 10M-doc Zipfian index) the same way.

N>1 (torchrun, one rank per GPU): the corpus is sharded by contiguous 64K-row level ranges (strong scaling);
every rank calls the same C-ABI search with the same batch, and the LIBRARY enqueues the exchange on its search stream
(ssb_comm_init: ncclAllGather of the packed top-k keys + G*k -> k merge, count all-reduce; hybrid: RRF after the merge).

After the timed regions rank 0 checks the (merged) top-10 of 64 vector + 64 BM25 queries against the CPU oracle and
reports "parity_check": {"n": 128, "mismatches": 0} — at every N.

--impl reference: times the CPU restatement of the reference path (oracle/, kind "port": the Rust reference
cannot be built here) on the host cores for the same metric / config.

Every timed loop runs --warmup untimed and exactly --steps timed steps.  --dump-outputs DIR writes what each timed
device path returned in its last timed step (top-10 doc ids, scores and counts) as DIR/<name>.npy; all inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it

import numpy as np  # noqa: E402
import torch  # noqa: E402

C2_ROWS, C2_DIMS, TOPK = 1_000_000, 768, 10
C3_DOCS, C3_VOCAB = 10_000_000, 1_000_000


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--batch", type=int, default=256, help="vector queries per step")
    p.add_argument("--rows", type=int, default=C2_ROWS)
    p.add_argument("--dims", type=int, default=C2_DIMS)
    p.add_argument("--sections", default="vector,int8,bm25,hybrid,c5,phrase,parity")
    p.add_argument("--int8-batch", type=int, default=1024, help="queries per step of the int8 (ScalarQuantizationI8) section")
    p.add_argument("--bm25-docs", type=int, default=C3_DOCS)
    p.add_argument("--bm25-batch", type=int, default=4096, help="lexical queries per step")
    p.add_argument("--hybrid-docs", type=int, default=5_000_000)
    p.add_argument("--phrase-docs", type=int, default=2_000_000, help="docs of the phrase-query section's corpus (with token positions)")
    p.add_argument("--c5-docs", type=int, default=10_000_000, help="C5: docs AND vectors of the sharded hybrid index")
    p.add_argument("--parity-queries", type=int, default=64, help="queries per path of the post-run oracle check")
    p.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of each cpu_baseline sample")
    p.add_argument("--vector-kernel", default="both", choices=["both", "all", "ffma", "tc", "tc64", "tcb", "tcb64", "tcb256", "filt", "filt256", "filt256p"],
                   help="FP32 FFMA2 scan, tcgen05 scans, or both = ffma + tcb + tcb256 (headline = the fastest: what AUTO picks)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the results of the last timed step of every device path as DIR/<name>.npy (--impl b200)")
    return p.parse_args()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def tensor_peak():
    """dense bf16 TFLOP/s: the burst figure (kernel timed alone) of MEASURED_PEAKS.json, else the nominal 2250."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops"]), "measured (burst)"
    except Exception:
        return 2250.0, "nominal"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  In-process NVML polling
    (nvidia_ml_py) every 10 ms; falls back to an `nvidia-smi -lms` child process.  (The first version polled nvidia-smi with
    power.draw in the query: each sample stalled kernel launches for milliseconds and the device-resident `value`, measured
    with the sampler running, came out slower than the e2e number measured without it.)"""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index: int):
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop = False
        self.p = None
        self.th = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid))
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def poll():
                while not self._stop:
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.mx.append(mx)
                        r = int(get_reasons(h))
                        for name, bit in self.REASONS:
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                    time.sleep(0.01)
            self.th = threading.Thread(target=poll, daemon=True)
            self.th.start()
        except Exception:
            self._start_smi(gpu_index)

    def _start_smi(self, gpu_index):
        q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def has_samples(self):
        if self.th is not None:
            return len(self.sm) > 0
        try:
            return self.p is None or os.path.getsize(self.f.name) > 0
        except OSError:
            return True

    def stop(self):
        if self.th is not None:
            self._stop = True
            self.th.join(timeout=2)
        elif self.p is not None:
            time.sleep(0.15)
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush()
            self.f.seek(0)
            for line in self.f:
                c = [x.strip() for x in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    self.sm.append(float(c[1])); self.mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            os.unlink(self.f.name)
        if not self.sm:
            return None
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.mx)), "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def dist_setup(n):
    if n <= 1:
        return 0, 1
    # NCCL's INFO log (communicator size, transport) goes to stdout, which main() has already re-pointed at stderr: rank 0's
    # stdout carries exactly one JSON line, and the driver can still read the rank count from the log
    os.environ.setdefault("NCCL_DEBUG", "INFO")
    os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", n))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    import datetime
    dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=1800))
    return rank, world


def timed_steps(fn, steps, warmup, world, sampler=None):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, device time, max over ranks.
    With a clock sampler, extra untimed warm-up steps keep the GPU under load until nvidia-smi delivers its first sample."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if sampler is not None and world == 1:
        t_end = time.perf_counter() + 3.0
        while not sampler.has_samples() and time.perf_counter() < t_end:
            fn()
            torch.cuda.synchronize()
    elif world > 1:
        # every rank must issue the same number of collectives: a FIXED number of extra untimed steps keeps the GPUs under
        # load while rank 0's nvidia-smi sampler starts (a rank-dependent loop here deadlocks the all-gather)
        for _ in range(100):
            fn()
        torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms


# --dump-outputs: name -> array of what a timed path returned in its last timed step (rank 0; None = not dumping)
_OUTPUTS = None
DUMP_BYTES = 60 << 20       # row-sampled above this, so that the .npy files stay under 64 MB in all


def keep_keys(name, keys_dev, n, counts_dev=None):
    """Record the top-10 that a device-resident search left as packed keys (u64 = ordered(score) << 32 | 0xFFFFFFFF - doc_id,
    0 = empty slot; include/seekstorm_b200.h) as doc ids (float64, -1 = empty) and scores (float32, 0 = empty)."""
    if _OUTPUTS is None:
        return
    k = keys_dev[:n, :TOPK].cpu().numpy().view(np.uint64)
    o = (k >> np.uint64(32)).astype(np.uint32)
    bits = np.where(o & np.uint32(0x80000000), o & np.uint32(0x7FFFFFFF), ~o).astype(np.uint32)
    doc = np.uint32(0xFFFFFFFF) - (k & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    _OUTPUTS[name + "_ids"] = np.where(k == 0, -1.0, doc.astype(np.float64))
    _OUTPUTS[name + "_scores"] = np.where(k == 0, np.float32(0), bits.view(np.float32))
    if counts_dev is not None:
        _OUTPUTS[name + "_counts"] = counts_dev[:n].cpu().numpy().astype(np.float64)


def keep_hits(name, hits, n_hits):
    """Record host hits (ssb_hit [nq * 10], n_hits [nq]) as doc ids (float64, -1 = empty) and scores (float32, 0 = empty)."""
    if _OUTPUTS is None:
        return
    h = hits[:len(n_hits) * TOPK].reshape(len(n_hits), TOPK)
    full = np.arange(TOPK)[None, :] < n_hits[:, None]
    _OUTPUTS[name + "_ids"] = np.where(full, h["doc_id"].astype(np.float64), -1.0)
    _OUTPUTS[name + "_scores"] = np.where(full, h["score"], np.float32(0))


def write_outputs(path):
    """DIR/<name>.npy for every recorded array.  Above DUMP_BYTES in all, every array keeps the same fraction of its rows (queries),
    chosen by a fixed seed, so that the files of two runs still line up."""
    os.makedirs(path, exist_ok=True)
    total = sum(v.nbytes for v in _OUTPUTS.values())
    frac = DUMP_BYTES / total if total > DUMP_BYTES else 1.0
    for name, v in _OUTPUTS.items():
        if frac < 1.0:
            v = v[np.sort(np.random.default_rng(0).choice(len(v), max(1, int(len(v) * frac)), replace=False))]
        np.save(os.path.join(path, name + ".npy"), v)


# ----------------------------------------------------------------------------------------------------------------
def vector_levels(rows, rank, world):
    from seekstorm_b200.parallel import level_range
    n_levels = (rows + 65535) // 65536
    return n_levels, level_range(n_levels, rank, world)


def gen_vector_level(level, rows, dims, device):
    from seekstorm_b200 import synth
    n = min(65536, rows - level * 65536)
    return synth.gen_vectors(n, dims, 1002 * 1000 + level, device)


KERNELS = {"ffma": (1, 16, "scan_ffma", "scan_ffma (TMA + packed FP32 FFMA2 + warp top-k)"),
           "tc": (2, 128, "scan_tc", "scan_tc (TMA + tcgen05 3xTF32 split, TMEM accumulators, TMEM-epilogue top-k)"),
           "tc64": (3, 64, "scan_tc", "scan_tc<64> (tcgen05 3xTF32, 64 queries per pass)"),
           "tcb": (4, 128, "scan_tc", "scan_tc (TMA + tcgen05 3xBF16 split, TMEM accumulators, TMEM-epilogue top-k)"),
           "tcb64": (5, 64, "scan_tc", "scan_tc<64> (tcgen05 3xBF16, 64 queries per pass)"),
           "tcb256": (6, 256, "scan_tc", "scan_tc<256> (tcgen05 3xBF16 over bf16 planes, 256 queries per pass: half the HBM bytes per query)"),
           # filter scan: ONE fp16 product over the 2-byte plane selects (proven margin) the <= 32 rows that can be in the top-10, refine
           # re-scores them with the f32 dot product; the result is the exact f32 top-k (DESIGN.md 3.2c)
           "filt": (7, 128, "scan_tc", "scan_tc<128, f16 filter> + refine_candidates (tcgen05 1xFP16 over the 2-byte plane, exact f32 re-scoring of <= 32 candidates per query)"),
           "filt256": (8, 256, "scan_tc", "scan_tc<256, f16 filter> + refine_candidates (256 queries per pass)"),
           "filt256p": (9, 256, "scan_tc", "scan_tc2 (256-query f16 filter on CTA pairs, tcgen05 cta_group::2) + refine_candidates")}
# DRAM traffic per corpus pass (dram__bytes_read.sum + dram__bytes_write.sum of ONE ncu --set full capture, divided by
# the passes in that launch, 1M x 768 corpus) from the committed captures under profiles/: traffic ~= algorithmic bytes
# (3.072 GB), i.e. no re-reads.
NCU = {"scan_ffma": {"traffic_per_pass": 3.0770e9, "source": "profiles/r02_scan_ffma.summary.txt"},   # 3.0734 GB read + 3.6 MB written, one pass of 16 queries
       # bf16 hi/lo corpus planes: (6.1655 GB read + 58.7 MB written) / 2 passes; 256-query tile: 3.1087 GB + 75.5 MB, one pass
       "scan_tc": {"traffic_per_pass": 3.1121e9, "source": "profiles/r02_scan_tc_bf16_planes_v1.summary.txt", "tensor_pipe_pct": 66.1},
       "tcb256": {"traffic_per_pass": 3.1842e9, "source": "profiles/r02_scan_tc_bf16_n256_v1.summary.txt", "tensor_pipe_pct": 84.2},
       # filter scan (fp16 plane): 128-query tile (3.0909 GB read + 60.8 MB written) / 2 passes; 256-query tile 1.5575 GB + 59.2 MB, one pass
       "filt": {"traffic_per_pass": 1.5759e9, "source": "profiles/r02_scan_tc_filter_v1.summary.txt", "tensor_pipe_pct": 45.2},
       "filt256": {"traffic_per_pass": 1.6167e9, "source": "profiles/r02_scan_tc_filter_n256_v1.summary.txt", "tensor_pipe_pct": 62.1},
       # scan_tc2 (CTA pairs, 256 queries): 1.5575 GB read + 58.9 MB written in one pass of 355.5 us under ncu
       "filt256p": {"traffic_per_pass": 1.6164e9, "source": "profiles/r02_scan_tc2_filter_pair.summary.txt", "tensor_pipe_pct": 64.3},
       # int8 full scan of 1M x 768, 1024 queries = 8 passes in one launch: (6.2222 GB read + 219.8 MB written) / 8
       "scan_tc_i8": {"traffic_per_pass": 0.8052e9, "source": "profiles/r02_scan_tc_i8.summary.txt"},
       # lex_score<OR>, C3 10M docs, 4096 queries, Topk: 6.8986 GB read + 60.6 MB written (random 32-byte sector probes of the
       # bitmap sectors and the coarse tables on top of the 1.5 GB the algorithm names)
       "lex_score": {"traffic": 6.9592e9, "source": "profiles/r02_lex_score_v6.summary.txt"}}


def measure_vector_kernel(a, ix, kname, q_host, q_dev, keys, local_rows, rank, world, dev, want_clocks):
    kid, qt, kshort, klong = KERNELS[kname]
    ix.set_vector_kernel(kid)
    # ---- value: device-resident hot path.  N>1: the same call is a collective — the library enqueues the NCCL all-gather of
    # the packed keys and the merge behind the per-rank scan (ssb_comm_init), every rank ends up with the global top-k ----
    def step_dev():
        ix.search_vector_keys(q_dev, TOPK, keys)
    step_dev(); torch.cuda.synchronize()
    sampler = ClockSampler(dev.index) if want_clocks else None
    ms = timed_steps(step_dev, a.steps, a.warmup, world, sampler)
    keep_keys(f"vector_{kname}", keys, a.batch)
    clocks = sampler.stop() if sampler else None
    kern_ns = []
    for _ in range(5):       # duration of the dominant kernel: CUDA events the library records around that launch
        step_dev(); torch.cuda.synchronize()
        kern_ns.append(ix.last_stats()["dominant_kernel_ns"])
    launches = ix.last_stats()["kernel_launches"]
    passes = (a.batch + qt - 1) // qt
    # ---- e2e: the reference-facing call with HOST buffers (H2D queries, D2H hits inside the timed region), on every rank ----
    q_np = q_host.numpy()
    hits_buf, nh_buf = ix.hits_buffer(a.batch * TOPK), np.zeros(a.batch, dtype=np.uint32)

    def step_e2e():
        ix.search_vector_raw(q_np, TOPK, hits_buf, nh_buf)     # ssb_search_vector: host queries in, host hits out
    ms_e2e = timed_steps(step_e2e, a.steps, a.warmup, world)
    fallbacks = ix.last_stats().get("filter_fallbacks", 0)       # queries of the last e2e call that took the exact fallback scan
    peak, peak_kind = peaks()
    kern_ms = float(np.median(kern_ns)) / 1e6 if kern_ns and min(kern_ns) > 0 else None
    filt = kname.startswith("filt")
    # per launch (one launch = all passes of the batch).  SURVEY 8(d) counts rows*dims*4 per pass for an f32 scan; the filter scan's own
    # algorithm only has to stream the 2-byte plane, so ITS roofline is counted on rows*dims*2 (the f32-equivalent figure is reported beside it)
    alg_bytes = float(local_rows) * a.dims * (2 if filt else 4) * passes
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9 if kern_ms else None
    ncu = NCU.get(kname, NCU.get(kshort, {}))
    tensor = None
    if kshort == "scan_tc" and kern_ms:
        # every f32 product is three bf16 MMAs (hi*hi + hi*lo + lo*hi): executed flops = 3 x the algorithmic 2*rows*dims*queries
        tpeak, tkind = tensor_peak()
        alg_tf = 2.0 * local_rows * a.dims * qt * passes / (kern_ms / 1e3) / 1e12
        nprod = 1 if filt else 3
        tensor = {"algorithmic_tflops": alg_tf, "executed_tflops": nprod * alg_tf, "peak": tpeak, "peak_kind": tkind,
                  "frac_executed": nprod * alg_tf / tpeak, "tensor_pipe_pct_ncu": ncu.get("tensor_pipe_pct")}
    return {
        "value": a.batch * a.steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / a.steps,
        "e2e": {"value": a.batch * a.steps / (ms_e2e / 1e3), "unit": "queries/s", "ms_per_step": ms_e2e / a.steps,
                "h2d_bytes_per_step": a.batch * a.dims * 4, "d2h_bytes_per_step": a.batch * 32 * 8},
        "gpu_launches": int(launches) * a.steps, "queries_per_pass": qt, "passes_per_step": passes, "kernel_desc": klong,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None,
                     "traffic": (ncu["traffic_per_pass"] * passes * local_rows / 1e6) if (ncu and ncu.get("traffic_per_pass") and a.dims == C2_DIMS) else None,
                     "traffic_source": ncu.get("source"), "peak_kind": f"of {peak_kind}", "kernel": kshort, "kernel_ms": kern_ms,
                     "algorithmic_bytes_per_launch": alg_bytes, "tensor": tensor,
                     **({"f32_equivalent_gbs": float(local_rows) * a.dims * 4 * passes / (kern_ms / 1e3) / 1e9 if kern_ms else None,
                         "note": "filter scan: streams rows*dims*2 bytes per pass (fp16 plane) + <= 32 f32 rows per query in the refine step; "
                                 "achieved/frac are counted on the 2-byte plane, f32_equivalent_gbs is the SURVEY 8(d) figure rows*dims*4/t"} if filt else {})},
        "filter_fallbacks": int(fallbacks) if filt else None,
        "clocks": clocks,
    }


def best_hbm_variant(kernels: dict):
    """Among the measured scan variants, the one that sits highest on the HBM roofline (the headline is the FASTEST variant, which at 256
    queries per pass is bound by the tensor pipe / shared memory rather than by HBM): {"kernel", "frac", "achieved", "value", "kernel_ms"}."""
    best = None
    for name, r in kernels.items():
        rf = (r or {}).get("roofline") or {}
        if rf.get("frac") is None:
            continue
        if best is None or rf["frac"] > best["frac"]:
            best = {"kernel": name, "frac": rf["frac"], "achieved": rf.get("achieved"), "unit": rf.get("unit"), "value": r.get("value"),
                    "kernel_ms": rf.get("kernel_ms")}
    return best


def bench_vector(a, rank, world, out):
    from seekstorm_b200 import Index, VectorSimilarity, synth
    from seekstorm_b200.parallel import init_shard_comm
    dev = torch.device("cuda", torch.cuda.current_device())
    ix = Index(dev.index, vector_dims=a.dims, vector_similarity=VectorSimilarity.Cosine, max_batch=max(a.batch, 16))
    ix.set_stream(torch.cuda.current_stream().cuda_stream)
    if world > 1:
        init_shard_comm(ix)
    n_levels, mine = vector_levels(a.rows, rank, world)
    local_rows = 0
    ix.reserve_vectors(sum(min(65536, a.rows - lv * 65536) for lv in mine))
    for lv in mine:
        r = gen_vector_level(lv, a.rows, a.dims, dev)
        ix.add_vector_level(lv, r)
        local_rows += r.shape[0]
        del r
    q_host = synth.gen_vectors(a.batch, a.dims, 2002, "cpu").pin_memory()
    q_dev = q_host.to(dev)
    keys = torch.zeros((a.batch, 32), dtype=torch.int64, device=dev)
    names = ["ffma", "tcb", "tcb256", "filt", "filt256", "filt256p"] if a.vector_kernel in ("both", "all") else [a.vector_kernel]
    res = {k: measure_vector_kernel(a, ix, k, q_host, q_dev, keys, local_rows, rank, world, dev, rank == 0) for k in names}
    # batch-size sweep through the reference-facing call (host buffers, AUTO kernel choice): latency at batch 1 .. 256
    sweep = {}
    if world == 1:
        ix.set_vector_kernel(0)
        for bs in (1, 8, 64, 256):
            if bs > a.batch:
                continue
            qn = q_host.numpy()[:bs].copy()
            hb, nb = ix.hits_buffer(bs * TOPK), np.zeros(bs, dtype=np.uint32)

            def step_b():
                ix.search_vector_raw(qn, TOPK, hb, nb)
            per = timed_steps(step_b, a.steps, a.warmup, world) / a.steps
            sweep[str(bs)] = {"ms_per_call": per, "queries_per_s": bs / (per / 1e3)}
    best = max(names, key=lambda k: res[k]["value"])      # headline = what SSB_VEC_KERNEL_AUTO picks for this batch size
    r = res[best]
    out.update({
        "metric": "queries/sec at top-10 (1M x 768 f32 cosine brute-force kNN)", "value": r["value"], "unit": "queries/s",
        "ms_per_step": r["ms_per_step"], "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C2 brute-force cosine kNN: {a.rows} x {a.dims} f32, top-{TOPK}, batch {a.batch} queries/step "
                               f"({r['passes_per_step']} corpus passes of {r['queries_per_pass']} queries)",
                   "l2": "inputs larger than L2 (corpus %.2f GB per GPU)" % (local_rows * a.dims * 4 / 1e9),
                   "parallelism": f"64K-row levels sharded over {world} GPU(s)", "kernel": r["kernel_desc"]},
        "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "roofline": r["roofline"], "clocks": r["clocks"],
        "batch_sweep_e2e": sweep,
        "kernels": {{"ffma": "scan_ffma", "tc": "scan_tc_tf32", "tc64": "scan_tc_tf32_n64", "tcb": "scan_tc_bf16", "tcb64": "scan_tc_bf16_n64", "tcb256": "scan_tc_bf16_n256",
                     "filt": "scan_tc_f16_filter", "filt256": "scan_tc_f16_filter_n256", "filt256p": "scan_tc2_f16_filter_n256_pair"}[k]:
                    {kk: vv for kk, vv in res[k].items() if kk != "kernel_desc"} for k in names},
    })
    try:   # the same corpus pass at its most HBM-efficient tile, next to the (faster) headline kernel
        out["roofline"] = dict(out["roofline"], best_hbm_fraction_variant=best_hbm_variant(out["kernels"]))
    except Exception:  # pragma: no cover
        pass
    return ix, q_host


def bench_vector_int8(a, rank, world):
    """C2 corpus with Cosine + ScalarQuantizationI8 (SURVEY §8f row 2): int8 corpus, tcgen05 kind::i8 scan, exact scores."""
    from seekstorm_b200 import Index, VectorSimilarity, synth
    from seekstorm_b200.parallel import init_shard_comm
    dev = torch.device("cuda", torch.cuda.current_device())
    nb = a.int8_batch
    ix = Index(dev.index, vector_dims=a.dims, vector_similarity=VectorSimilarity.Cosine, max_batch=max(nb, 16), vector_quantization=1)
    ix.set_stream(torch.cuda.current_stream().cuda_stream)
    if world > 1:
        init_shard_comm(ix)
    n_levels, mine = vector_levels(a.rows, rank, world)
    local_rows = 0
    ix.reserve_vectors(sum(min(65536, a.rows - lv * 65536) for lv in mine))
    for lv in mine:
        r = gen_vector_level(lv, a.rows, a.dims, dev)
        ix.add_vector_level(lv, r)
        local_rows += r.shape[0]
        del r
    q_host = synth.gen_vectors(nb, a.dims, 2002, "cpu").pin_memory()
    q_dev = q_host.to(dev)
    keys = torch.zeros((nb, 32), dtype=torch.int64, device=dev)

    def step_dev():
        ix.search_vector_keys(q_dev, TOPK, keys)
    step_dev(); torch.cuda.synchronize()
    ms = timed_steps(step_dev, a.steps, a.warmup, world)
    keep_keys("int8", keys, nb)
    kern_ns = []
    for _ in range(5):
        step_dev(); torch.cuda.synchronize()
        kern_ns.append(ix.last_stats()["dominant_kernel_ns"])
    launches = ix.last_stats()["kernel_launches"]
    q_np = q_host.numpy()
    hits_buf, nh_buf = ix.hits_buffer(nb * TOPK), np.zeros(nb, dtype=np.uint32)

    def step_e2e():
        ix.search_vector_raw(q_np, TOPK, hits_buf, nh_buf)
    ms_e2e = timed_steps(step_e2e, a.steps, a.warmup, world)
    sweep = {}
    if world == 1:
        for bs in (1, 128, 256):
            qn = q_np[:bs].copy()
            hb, nbuf = ix.hits_buffer(bs * TOPK), np.zeros(bs, dtype=np.uint32)

            def step_b():
                ix.search_vector_raw(qn, TOPK, hb, nbuf)
            per = timed_steps(step_b, a.steps, a.warmup, world) / a.steps
            sweep[str(bs)] = {"ms_per_call": per, "queries_per_s": bs / (per / 1e3)}
    peak, peak_kind = peaks()
    passes = (nb + 127) // 128
    kern_ms = float(np.median(kern_ns)) / 1e6 if kern_ns and min(kern_ns) > 0 else None
    alg_bytes = float(local_rows) * a.dims * 1 * passes
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9 if kern_ms else None
    ix.close()
    return {
        "metric": "queries/sec at top-10 (1M x 768 cosine, ScalarQuantizationI8 brute-force kNN)",
        "value": nb * a.steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / a.steps, "dtype": "i8 (int32 accumulate, exact)",
        "config": {"workload": f"C2 corpus quantised to int8 (Cosine + ScalarQuantizationI8): {a.rows} x {a.dims}, top-{TOPK}, "
                               f"batch {nb} queries/step ({passes} corpus passes of 128 queries)",
                   "kernel": "scan_tc<128, i8> (tcgen05 kind::i8, TMEM s32 accumulators)"},
        "e2e": {"value": nb * a.steps / (ms_e2e / 1e3), "unit": "queries/s", "ms_per_step": ms_e2e / a.steps,
                "h2d_bytes_per_step": nb * a.dims * 4, "d2h_bytes_per_step": nb * 32 * 8},
        "gpu_launches": int(launches) * a.steps, "batch_sweep_e2e": sweep,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                     "traffic": (NCU["scan_tc_i8"]["traffic_per_pass"] * passes * local_rows / 1e6) if a.dims == C2_DIMS else None,
                     "traffic_source": NCU["scan_tc_i8"]["source"],
                     "peak_kind": f"of {peak_kind}", "kernel": "scan_tc_i8", "kernel_ms": kern_ms,
                     "algorithmic_bytes_per_launch": alg_bytes},
    }


def bench_vector_int8_variants(a, rank, world):
    """SURVEY 8(f) row 2, the other int8 quantisers on the int8 tcgen05 scan: TurboQuantI8 (1M x 768 cosine: rows are next_power_of_two(768) =
    1024 code bytes) and the affine Euclidean SQ of integer-valued data (SIFT-like 1M x 128).  Device-resident QPS + the scan's roofline."""
    from seekstorm_b200 import Index, VectorSimilarity, synth
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {}
    peak, peak_kind = peaks()
    nb = a.int8_batch
    for name in ("turboquant_i8", "affine_sq_i8"):
        dims = a.dims if name == "turboquant_i8" else 128
        if name == "turboquant_i8":
            ix = Index(dev.index, vector_dims=dims, vector_similarity=VectorSimilarity.Cosine, max_batch=max(nb, 16), vector_quantization=2)
            dim2 = 1
            while dim2 < dims:
                dim2 *= 2
            ix.set_turboquant_mask(np.where(np.random.default_rng(1234).random(dim2) < 0.5, 1.0, -1.0).astype(np.float32))
            row_bytes = dim2
        else:
            ix = Index(dev.index, vector_dims=dims, vector_similarity=VectorSimilarity.Euclidean, max_batch=max(nb, 16), vector_quantization=1)
            row_bytes = dims
        ix.set_stream(torch.cuda.current_stream().cuda_stream)
        ix.reserve_vectors(a.rows)
        for lv in range((a.rows + 65535) // 65536):
            r = gen_vector_level(lv, a.rows, dims, dev)
            if name == "affine_sq_i8":
                r = (r.abs() * (45.0 * dims ** 0.5)).round().clamp_(0, 255)       # integer-valued 0..255 rows (SIFT-like)
            ix.add_vector_level(lv, r)
            del r
        q = synth.gen_vectors(nb, dims, 2002, "cpu")
        if name == "affine_sq_i8":
            q = (q.abs() * (45.0 * dims ** 0.5)).round().clamp_(0, 255)
        q_dev = q.to(dev)
        keys = torch.zeros((nb, 32), dtype=torch.int64, device=dev)

        def step_dev():
            ix.search_vector_keys(q_dev, TOPK, keys)
        step_dev(); torch.cuda.synchronize()
        ms = timed_steps(step_dev, a.steps, a.warmup, world)
        keep_keys(name, keys, nb)
        kern_ns = []
        for _ in range(3):
            step_dev(); torch.cuda.synchronize()
            kern_ns.append(ix.last_stats()["dominant_kernel_ns"])
        passes = (nb + 127) // 128
        kern_ms = float(np.median(kern_ns)) / 1e6 if kern_ns and min(kern_ns) > 0 else None
        alg = float(a.rows) * row_bytes * passes
        out[name] = {"value": nb * a.steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / a.steps,
                     "config": {"workload": f"{a.rows} x {dims}, top-{TOPK}, batch {nb} queries/step ({passes} passes of 128), {row_bytes} code bytes per row"},
                     "roofline": {"bound": "hbm", "achieved": alg / (kern_ms / 1e3) / 1e9 if kern_ms else None, "peak": peak, "unit": "GB/s",
                                  "frac": alg / (kern_ms / 1e3) / 1e9 / peak if kern_ms else None, "peak_kind": f"of {peak_kind}", "kernel": "scan_tc_i8 (scaled epilogue)",
                                  "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": alg, "traffic": None}}
        ix.close()
    return out


def cpu_vector_int8_baseline(a, seconds):
    """Restated reference CPU path for Cosine + SQ-I8 (dot_i8 over the int8 corpus, linear top-k), one query per thread."""
    from oracle import oracle as O
    from seekstorm_b200 import synth
    cores = os.cpu_count() or 1
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    rows = np.empty((a.rows, a.dims), dtype=np.int8)
    sl = 65536

    def quant(lv):
        r = gen_vector_level(lv, a.rows, a.dims, dev).cpu().numpy()
        rows[lv * sl: lv * sl + r.shape[0]] = O.quantize_rows_i8(r)
    for lv in range((a.rows + sl - 1) // sl):
        quant(lv)
    qs = synth.gen_vectors(64, a.dims, 2002, "cpu").numpy()
    q8 = O.quantize_rows_i8(qs)
    O.search_vector_i8(rows, q8[0], TOPK)
    done = [0] * cores
    stop = time.perf_counter() + seconds
    nxt = [0]
    lock = threading.Lock()

    def work(i):
        while time.perf_counter() < stop:
            with lock:
                j = nxt[0]; nxt[0] += 1
            O.search_vector_i8(rows, q8[j % len(q8)], TOPK)
            done[i] += 1
    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
    [t.start() for t in th]; [t.join() for t in th]
    dt = time.perf_counter() - t0
    n_done = sum(done)
    return {"value": n_done / dt, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{n_done} queries, full {a.rows}x{a.dims} int8 corpus, {cores} threads (one query each), {dt:.1f}s"}


def cpu_vector_baseline(a, seconds):
    """The restated reference CPU path (oracle: exhaustive scan, 8-lane FMA dot as dot_f32_avx2, linear top-k), all
    host threads, on a bounded sample of the C2 queries."""
    from oracle import oracle as O
    from seekstorm_b200 import synth
    cores = os.cpu_count() or 1
    rows = np.empty((a.rows, a.dims), dtype=np.float32)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    for lv in range((a.rows + 65535) // 65536):
        r = gen_vector_level(lv, a.rows, a.dims, dev)
        r = r / r.norm(dim=1, keepdim=True)
        rows[lv * 65536: lv * 65536 + r.shape[0]] = r.cpu().numpy()
    # spread the corpus pages over the NUMA nodes: re-copy it with one first-touching worker per slice (the single
    # allocating thread above would otherwise place all 3 GB on its own node and cap the scan at one socket's bandwidth)
    rows2 = np.empty_like(rows)
    sl = max(1, (a.rows + cores - 1) // cores)

    def touch(i):
        rows2[i * sl:(i + 1) * sl] = rows[i * sl:(i + 1) * sl]
    tt = [threading.Thread(target=touch, args=(i,)) for i in range(cores)]
    [t.start() for t in tt]; [t.join() for t in tt]
    rows = rows2
    qs = synth.gen_vectors(a.batch, a.dims, 2002, "cpu").numpy()
    qn = [O.normalize(q) for q in qs]
    O.search_vector(rows, qn[0], TOPK, O.SIM_COSINE, lanes8=True, n_threads=cores)  # warm (page in the corpus)
    # one worker per core, each answering whole queries single-threaded (8-lane FMA dot, linear top-k): the
    # throughput-optimal arrangement of the reference's per-shard scan on this host
    samples = []
    for _ in range(2):
        done = [0] * cores
        stop = time.perf_counter() + seconds / 2
        nxt = [0]
        lock = threading.Lock()

        def work(i):
            _pin(i)
            while time.perf_counter() < stop:
                with lock:
                    j = nxt[0]; nxt[0] += 1
                O.search_vector(rows, qn[j % len(qn)], TOPK, O.SIM_COSINE, lanes8=True, n_threads=1)
                done[i] += 1
        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
        [t.start() for t in th]; [t.join() for t in th]
        dt = time.perf_counter() - t0
        samples.append(sum(done) / dt)
    best = max(samples)
    return {"value": best, "unit": "queries/s", "cores": cores, "kind": "port", "samples": samples,
            "scan_gb_per_s": best * a.rows * a.dims * 4 / 1e9,
            "sample": f"2 x {seconds / 2:.0f}s, cycling the {a.batch} C2 queries over the full {a.rows}x{a.dims} corpus (first-touched per thread slice), "
                      f"{cores} pinned threads (one query each); CPU restatement of the reference scan (no Rust toolchain here), not the reference binary"}


# ----------------------------------------------------------------------------------------------------------------
def build_bm25(a, rank, world, dev, n_docs, seed, vector_dims=0):
    """Lexical index of `n_docs` docs (this rank's contiguous level range); N>1: library-owned NCCL communicator + index-wide df."""
    from seekstorm_b200 import Index, VectorSimilarity, synth
    from seekstorm_b200.parallel import level_range, init_shard_comm
    ix = Index(dev.index if dev.type == "cuda" else 0, max_batch=max(a.bm25_batch, 1024), vector_dims=vector_dims,
               vector_similarity=VectorSimilarity.Cosine)
    ix.set_stream(torch.cuda.current_stream().cuda_stream)
    if world > 1:
        init_shard_comm(ix)
    n_levels = (n_docs + 65535) // 65536
    mine = level_range(n_levels, rank, world)
    len_sum = torch.zeros(1, dtype=torch.int64, device=dev)
    for lv in synth.gen_lexical_corpus(n_docs, C3_VOCAB, seed, dev, level_ids=mine):
        ix.add_synth_level(lv)
        len_sum += lv.len_sum_normalized
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(len_sum)
    ix.commit(n_docs, int(len_sum.item()))
    if world > 1:
        ix.sync_df()
    return ix, int(len_sum.item())


def bm25_queries(n, seed=2003):
    from seekstorm_b200 import synth
    qs = synth.gen_queries(n, seed, 20, 100000, (2, 3, 4), (0.4, 0.4, 0.2))
    return [[int(k) for k in synth.term_keys_np(np.array(q, dtype=np.int64))] for q in qs]


def _bm25_filter_variants(a, ix, qk, out_keys, world, dev):
    """SURVEY 8(f) row 4: the C3 OR queries behind a facet range filter that half of the docs pass (is_facet_filter on every candidate; filtered
    queries are scored and counted doc by doc in lex_generic) — 1024 queries per step, Topk and TopkCount."""
    from seekstorm_b200 import FacetFilter, QueryType, ResultType
    price = np.random.default_rng(1007).integers(0, 1000, a.bm25_docs, dtype=np.uint32)
    ix.set_facets({"price": price})
    nf = min(1024, len(qk))
    bf, keep_f = ix._lex_batch(qk[:nf], QueryType.Union, None, [[FacetFilter("price", 0, 500)]] * nf)
    cnt_dev = torch.zeros(nf, dtype=torch.int64, device=dev)
    res = {}
    for name, rt_ in (("or_topk_facet_filter", ResultType.Topk), ("or_topkcount_facet_filter", ResultType.TopkCount)):
        def step_f():
            ix.search_lexical_keys(bf, TOPK, rt_, out_keys, cnt_dev)
        msv = timed_steps(step_f, a.steps, a.warmup, world)
        keep_keys(f"bm25_{name}", out_keys, nf, cnt_dev if rt_ == ResultType.TopkCount else None)
        step_f(); torch.cuda.synchronize()
        sv = ix.last_stats()
        res[name] = {"value": nf * a.steps / (msv / 1e3), "unit": "queries/s", "kernel_ms": sv["dominant_kernel_ns"] / 1e6, "queries_per_step": nf,
                     "selectivity": 0.5, "kernel": "lex_score<.., HAS_NOT> (Topk: filter on the exact-score survivors) / lex_generic (counts: every match tested)"}
    ix.set_facets({})
    return res


def bench_phrase(a, rank, world):
    """SURVEY 8(f) row 4, QueryType::Phrase: a Zipf corpus of the C3 law with token positions (2 M docs by default), 1024 phrases of 2-3 frequent
    terms per step; intersection of the phrase's terms + the position check per candidate (lex_generic).  Device-resident QPS."""
    from seekstorm_b200 import Index, QueryType, ResultType, synth
    dev = torch.device("cuda", torch.cuda.current_device())
    n = a.phrase_docs
    ix = Index(dev.index, max_batch=1024)
    ix.set_stream(torch.cuda.current_stream().cuda_stream)
    ls, n_pos = 0, 0
    t0 = time.perf_counter()
    for lv in synth.gen_lexical_corpus(n, C3_VOCAB, 1006, dev, with_positions=True):
        ix.add_synth_level(lv)
        ls += lv.len_sum_normalized
        n_pos += int(lv.positions.numel())
    ix.commit(n, ls)
    build_s = time.perf_counter() - t0
    rng = np.random.default_rng(2006)
    phrases = [[int(x) for x in np.floor(np.exp(rng.uniform(0, np.log(300), int(rng.integers(2, 4)))))] for _ in range(1024)]
    qk = [[int(k) for k in synth.term_keys_np(np.array(p, dtype=np.int64))] for p in phrases]
    b, keep = ix._lex_batch(qk, QueryType.Phrase)
    out_keys = torch.zeros((len(qk), 32), dtype=torch.int64, device=dev)
    cnt_dev = torch.zeros(len(qk), dtype=torch.int64, device=dev)
    res = {"config": {"workload": f"{n} docs Zipf(1) V={C3_VOCAB} with positions ({n_pos} tokens), {len(qk)} phrases/step of 2-3 terms, ranks log-uniform [1,300]",
                      "index_build_s": build_s}}
    for name, rt_ in (("topk", ResultType.Topk), ("topkcount", ResultType.TopkCount)):
        def step():
            ix.search_lexical_keys(b, TOPK, rt_, out_keys, cnt_dev)
        ms = timed_steps(step, a.steps, a.warmup, world)
        keep_keys(f"phrase_{name}", out_keys, len(qk), cnt_dev if rt_ == ResultType.TopkCount else None)
        step(); torch.cuda.synchronize()
        sv = ix.last_stats()
        res[name] = {"value": len(qk) * a.steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / a.steps, "kernel_ms": sv["dominant_kernel_ns"] / 1e6,
                     "postings_visited": sv.get("postings_visited"), "kernel": "lex_generic (intersection + phrase predicate)"}
    res["matching_phrases"] = int((cnt_dev > 0).sum().item())
    ix.close()
    return res


def bench_bm25(a, rank, world, keep_index=False, vector_dims=0):
    from seekstorm_b200 import QueryType, ResultType
    dev = torch.device("cuda", torch.cuda.current_device())
    t0 = time.perf_counter()
    ix, len_sum = build_bm25(a, rank, world, dev, a.bm25_docs, 1003, vector_dims)
    build_s = time.perf_counter() - t0
    qk = bm25_queries(a.bm25_batch)
    b, keep = ix._lex_batch(qk, QueryType.Union)
    offs_dev = torch.from_numpy(keep[0].view(np.int32)).to(dev)
    keys_dev = torch.from_numpy(keep[1].view(np.int64)).to(dev)
    from seekstorm_b200._lib import SsbLexBatch
    b_dev = SsbLexBatch(len(qk), int(QueryType.Union), offs_dev.data_ptr(), keys_dev.data_ptr())
    out_keys = torch.zeros((len(qk), 32), dtype=torch.int64, device=dev)

    def step_dev():     # N>1: collective (all-gather + merge of the packed keys inside the library)
        ix.search_lexical_keys(b_dev, TOPK, ResultType.Topk, out_keys)
    ms = timed_steps(step_dev, a.steps, a.warmup, world)
    keep_keys("bm25", out_keys, len(qk))
    kern_ns = []
    for _ in range(3):
        step_dev(); torch.cuda.synchronize()
        kern_ns.append(ix.last_stats()["dominant_kernel_ns"])
    st = ix.last_stats()
    launches = st["kernel_launches"]

    hits_buf, nh_buf, cnt_buf = ix.hits_buffer(len(qk) * TOPK), np.zeros(len(qk), dtype=np.uint32), np.zeros(len(qk), dtype=np.uint64)

    def step_e2e():
        ix.search_lexical_raw(b, TOPK, ResultType.Topk, hits_buf, nh_buf, cnt_buf)   # ssb_search_lexical, host buffers
    ms_e2e = timed_steps(step_e2e, a.steps, a.warmup, world)
    # secondary modes on the same index / queries (device-resident, same timing rules): exact counts and AND
    variants = {}
    for name, qt_, rt_ in (("or_topkcount", QueryType.Union, ResultType.TopkCount), ("and_topkcount", QueryType.Intersection, ResultType.TopkCount),
                           ("and_topk", QueryType.Intersection, ResultType.Topk)):
        bv = SsbLexBatch(len(qk), int(qt_), offs_dev.data_ptr(), keys_dev.data_ptr())
        cnt_dev = torch.zeros(len(qk), dtype=torch.int64, device=dev)

        def step_v():
            ix.search_lexical_keys(bv, TOPK, rt_, out_keys, cnt_dev)
        msv = timed_steps(step_v, a.steps, a.warmup, world)
        keep_keys(f"bm25_{name}", out_keys, len(qk), cnt_dev if rt_ == ResultType.TopkCount else None)
        step_v(); torch.cuda.synchronize()
        sv = ix.last_stats()
        variants[name] = {"value": len(qk) * a.steps / (msv / 1e3), "unit": "queries/s", "kernel_ms": sv["dominant_kernel_ns"] / 1e6,
                          "algorithmic_bytes_per_launch": sv["algorithmic_bytes"]}
    if world == 1:
        try:
            variants.update(_bm25_filter_variants(a, ix, qk, out_keys, world, dev))
        except Exception as e:  # pragma: no cover
            variants["or_topk_facet_filter"] = {"error": repr(e)}
    peak, peak_kind = peaks()
    kern_ms = float(np.median(kern_ns)) / 1e6 if kern_ns and min(kern_ns) > 0 else None
    alg = st.get("algorithmic_bytes")
    res = {
        "metric": "queries/sec at top-10 (BM25 OR, block-max pruned, ResultType::Topk)", "value": len(qk) * a.steps / (ms / 1e3),
        "unit": "queries/s", "ms_per_step": ms / a.steps, "steps": a.steps, "dtype": "f32 scores / u16 postings",
        "config": {"workload": f"C3 BM25 OR top-{TOPK}: {a.bm25_docs} docs Zipf(1) V={C3_VOCAB}, {len(qk)} queries/step of 2-4 terms (40/40/20%), ranks log-uniform [20,1e5]",
                   "index_build_s": build_s, "l2": "posting arenas larger than L2 (12 B per posting: stream word, payload, f32 component; %.1f GB per GPU)" % (12 * 0.08 * a.bm25_docs / world / 1e6 / 1e3 * 1e3)},
        "e2e": {"value": len(qk) * a.steps / (ms_e2e / 1e3), "unit": "queries/s", "ms_per_step": ms_e2e / a.steps,
                "h2d_bytes_per_step": int(keep[0].nbytes + keep[1].nbytes), "d2h_bytes_per_step": len(qk) * (32 * 8 + 8)},
        "gpu_launches": int(launches) * a.steps, "variants": variants,
        "roofline": {"bound": "hbm", "achieved": (alg / (kern_ms / 1e3) / 1e9) if (alg and kern_ms) else None, "peak": peak, "unit": "GB/s",
                     "frac": (alg / (kern_ms / 1e3) / 1e9 / peak) if (alg and kern_ms) else None,
                     "traffic": NCU["lex_score"]["traffic"] if (a.bm25_docs == C3_DOCS and len(qk) == 4096 and world == 1) else None,
                     "traffic_source": NCU["lex_score"]["source"],
                     "peak_kind": f"of {peak_kind}", "kernel": "lex_score (+ lex_generic)", "kernel_ms": kern_ms,
                     "algorithmic_bytes_per_launch": alg, "postings_visited": st.get("postings_visited"), "probes": st.get("probes"),
                     "items_processed": st.get("items_processed"), "items_skipped": st.get("items_skipped")},
    }
    if keep_index:
        return res, ix
    ix.close()
    return res, None


def _add_vector_levels(ix, n_rows, rank, world, dev, seed_base):
    from seekstorm_b200 import synth
    n_levels, mine = vector_levels(n_rows, rank, world)
    local = 0
    ix.reserve_vectors(sum(min(65536, n_rows - lv * 65536) for lv in mine))
    for lv in mine:
        r = synth.gen_vectors(min(65536, n_rows - lv * 65536), C2_DIMS, seed_base * 1000 + lv, dev)
        ix.add_vector_level(lv, r)
        local += r.shape[0]
        del r
    return local


def _hybrid_steps(a, ix, qk, qv, world, name):
    from seekstorm_b200 import QueryType
    from seekstorm_b200._lib import check, lib
    import ctypes as C
    nq = len(qk)
    b, keep = ix.make_lex_batch(qk, QueryType.Union)
    hits, nh = ix.hits_buffer(nq * TOPK), np.zeros(nq, dtype=np.uint32)

    def step():
        check(lib().ssb_search_hybrid(ix._h, C.byref(b), qv.ctypes.data, TOPK, hits.ctypes.data, nh.ctypes.data))
    ms = timed_steps(step, a.steps, a.warmup, world)
    keep_hits(name, hits, nh)
    launches = ix.last_stats()["kernel_launches"]
    return ms, int(qv.nbytes + keep[0].nbytes + keep[1].nbytes), launches


def bench_hybrid(a, rank, world):
    """C4: SearchMode::Hybrid (BM25 OR top-10 + 768-d cosine top-10, RRF k=0.6) over 5M docs through ssb_search_hybrid with host
    buffers: the lexical and the vector search run concurrently on two streams, the RRF join runs on the host inside the library
    (search.rs:1962-2035); N>1: both lists are merged over the shards before the fusion."""
    from seekstorm_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    n_docs = a.hybrid_docs
    ix, _ = build_bm25(a, rank, world, dev, n_docs, 1004, vector_dims=C2_DIMS)
    local_rows = _add_vector_levels(ix, n_docs, rank, world, dev, 1005)
    nq = 1000
    qk = bm25_queries(nq, 2004)
    qv = synth.gen_vectors(nq, C2_DIMS, 2005, "cpu").numpy()
    ms, h2d, launches = _hybrid_steps(a, ix, qk, qv, world, "hybrid")
    ix.close()
    peak, peak_kind = peaks()
    passes = (nq + 255) // 256                                   # AUTO: filter scan, 256 queries per pass over the 2-byte plane
    alg = float(local_rows) * C2_DIMS * 2 * passes
    return {"metric": "queries/sec at top-10 (hybrid: BM25 OR + 768-d cosine, RRF)", "value": nq * a.steps / (ms / 1e3), "unit": "queries/s",
            "ms_per_step": ms / a.steps, "steps": a.steps,
            "config": {"workload": f"C4 hybrid: {n_docs} docs (Zipf lexical index + {n_docs} x {C2_DIMS} f32 vectors), {nq} queries/step, e2e through ssb_search_hybrid (host buffers)"},
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": nq * 32 * 16, "gpu_launches": int(launches) * a.steps,
            # the step is bounded below by the vector scan: 4 filter passes of 256 queries over the 7.7 GB fp16 plane (f32-equivalent: x2)
            "roofline": {"bound": "hbm", "achieved": alg / (ms / a.steps / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms / a.steps / 1e3) / 1e9 / peak, "peak_kind": f"of {peak_kind}", "kernel": "whole step (filter scan_tc + refine, lex_score overlapped, host RRF)",
                         "algorithmic_bytes_per_launch": alg, "f32_equivalent_gbs": 2 * alg / (ms / a.steps / 1e3) / 1e9}}


def bench_c5(a, rank, world, ix):
    """C5 (BASELINE config 5): the C3 lexical index (already on `ix`) + 10M x 768 vectors, sharded by level range over the N GPUs,
    BM25 + vector + RRF, NCCL top-k merge inside the library."""
    from seekstorm_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    n = a.c5_docs
    t0 = time.perf_counter()
    local_rows = _add_vector_levels(ix, n, rank, world, dev, 1006)
    build_s = time.perf_counter() - t0
    nq = 1000
    qk = bm25_queries(nq, 2003)
    qv_t = synth.gen_vectors(nq, C2_DIMS, 2006, "cpu").pin_memory()
    qv = qv_t.numpy()
    ms, h2d, launches = _hybrid_steps(a, ix, qk, qv, world, "c5")
    # vector-only on the same shards (device-resident, batch 256): the scan at C5 size
    q_dev = qv_t[:a.batch].to(dev)
    keys = torch.zeros((a.batch, 32), dtype=torch.int64, device=dev)

    def step_v():
        ix.search_vector_keys(q_dev, TOPK, keys)
    msv = timed_steps(step_v, a.steps, a.warmup, world)
    keep_keys("c5_vector", keys, a.batch)
    kern = []
    for _ in range(3):
        step_v(); torch.cuda.synchronize()
        kern.append(ix.last_stats()["dominant_kernel_ns"])
    peak, peak_kind = peaks()
    passes = (a.batch + 255) // 256 if a.batch > 128 else 1      # AUTO: filter scan (2-byte plane), 256 (128) queries per pass
    alg = float(local_rows) * C2_DIMS * 2 * passes
    kern_ms = float(np.median(kern)) / 1e6 if kern and min(kern) > 0 else None
    return {"metric": "queries/sec at top-10 (C5: 10M docs BM25 + 10M x 768 cosine, RRF hybrid, sharded)", "value": nq * a.steps / (ms / 1e3),
            "unit": "queries/s", "ms_per_step": ms / a.steps, "steps": a.steps,
            "config": {"workload": f"C5: {n} docs + {n} x {C2_DIMS} f32 vectors over {world} GPU(s) ({local_rows} rows on this rank), {nq} hybrid queries/step, e2e through ssb_search_hybrid",
                       "vector_build_s": build_s},
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": nq * 32 * 16, "gpu_launches": int(launches) * a.steps,
            "vector_only": {"value": a.batch * a.steps / (msv / 1e3), "unit": "queries/s", "batch": a.batch,
                            "roofline": {"bound": "hbm", "achieved": (alg / (kern_ms / 1e3) / 1e9) if kern_ms else None, "peak": peak, "unit": "GB/s",
                                         "frac": (alg / (kern_ms / 1e3) / 1e9 / peak) if kern_ms else None, "peak_kind": f"of {peak_kind}",
                                         "kernel": "scan_tc<256, f16 filter>", "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": alg,
                                         "f32_equivalent_gbs": (2 * alg / (kern_ms / 1e3) / 1e9) if kern_ms else None}}}


# ----------------------------------------------------------------------------------------------------------------
# post-run correctness evidence: merged top-10 of the first queries of each path against the CPU oracle (rank 0 checks; all
# ranks take part in the searches, which are collectives at N>1)
_ORACLE = {}


def oracle_lexical_index(a, n_docs, seed):
    """Exhaustive CPU oracle over the WHOLE corpus (all levels, generated on this rank's GPU and copied to the host once)."""
    from oracle import oracle as O
    from seekstorm_b200 import synth
    key = (n_docs, seed)
    if key in _ORACLE:
        return _ORACLE[key]
    dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    orc = O.OracleIndex()
    len_sum = 0
    for lv in synth.gen_lexical_corpus(n_docs, C3_VOCAB, seed, dev):
        orc.add_level(lv.to_numpy())
        len_sum += lv.len_sum_normalized
    orc.commit(n_docs, len_sum)
    _ORACLE[key] = orc
    return orc


def parity_vector(a, ix, q_host, rank, world):
    from oracle import oracle as O
    n = min(a.parity_queries, a.batch)
    ix.set_vector_kernel(0)
    got = ix.search_vector_batch(q_host.numpy()[:n], TOPK)        # collective at N>1: the global result on every rank
    if rank != 0:
        return None
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = np.empty((a.rows, a.dims), dtype=np.float32)
    for lv in range((a.rows + 65535) // 65536):
        r = gen_vector_level(lv, a.rows, a.dims, dev)
        rows[lv * 65536: lv * 65536 + r.shape[0]] = (r / r.norm(dim=1, keepdim=True)).cpu().numpy()
    bad = 0
    cores = os.cpu_count() or 1
    for i in range(n):
        want = O.search_vector(rows, O.normalize(q_host.numpy()[i]), TOPK, O.SIM_COSINE, n_threads=min(cores, 64))
        ok = len(got[i]) == len(want)
        for (gd, gs), (wd, ws) in zip(got[i], want):
            # north-star tolerance: 1e-4 relative on scores; ids identical except inside a tie closer than the tolerance
            if abs(gs - ws) > 1e-4 * max(abs(ws), 1e-6):
                ok = False
            if gd != wd and not any(gd == d2 for d2, _ in want) and abs(gs - want[-1][1]) > 1e-4 * max(abs(ws), 1e-6):
                ok = False
        bad += 0 if ok else 1
    return {"n": n, "mismatches": bad, "oracle": "exhaustive f32 scan (oracle/, 8-lane order off)", "tolerance": "ids identical (swaps only inside 1e-4 score ties), scores 1e-4 relative"}


def parity_bm25(a, ix, rank, world):
    from oracle import oracle as O
    from seekstorm_b200 import QueryType, ResultType
    n = a.parity_queries
    qk = bm25_queries(max(n, 1))[:n]
    got, counts = ix.search_lexical_batch(qk, QueryType.Union, TOPK, ResultType.TopkCount)
    got_and, counts_and = ix.search_lexical_batch(qk, QueryType.Intersection, TOPK, ResultType.TopkCount)
    if rank != 0:
        return None
    orc = oracle_lexical_index(a, a.bm25_docs, 1003)
    bad = 0
    for i, kq in enumerate(qk):
        want, tot = orc.search(kq, O.QUERY_UNION, TOPK, O.RESULT_TOPKCOUNT)
        wand, tand = orc.search(kq, O.QUERY_INTERSECTION, TOPK, O.RESULT_TOPKCOUNT)
        ok = got[i] == want and int(counts[i]) == tot and got_and[i] == wand and int(counts_and[i]) == tand
        bad += 0 if ok else 1
    return {"n": n, "mismatches": bad, "oracle": "exhaustive BM25 (oracle/)", "tolerance": "ids, ranks, scores and counts bit-exact; OR and AND of each query"}


def _pin(i):
    """Pin the calling worker thread to one core (threads stay on their NUMA node; the corpus was first-touched per slice)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        os.sched_setaffinity(0, {cpus[i % len(cpus)]})
    except Exception:
        pass


def cpu_bm25_baseline(a, seconds):
    """Reference-shaped CPU search (oracle pruned path: block-max ordered AND, union_docid_2-shaped 2-term OR, MAXSCORE for 3+
    terms) on the same index, one pinned worker thread per host core (the reference runs one task per shard, default shards =
    cores).  Two back-to-back samples so that box-to-box and run-to-run swings are visible in one record."""
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    orc = oracle_lexical_index(a, a.bm25_docs, 1003)
    qk = bm25_queries(a.bm25_batch)
    samples = []
    for _ in range(2):
        done = [0] * cores
        stop = time.perf_counter() + seconds / 2
        nxt = [0]
        lock = threading.Lock()

        def work(i):
            _pin(i)
            while time.perf_counter() < stop:
                with lock:
                    j = nxt[0]; nxt[0] += 1
                orc.search(qk[j % len(qk)], O.QUERY_UNION, TOPK, O.RESULT_TOPK, pruned=True)
                done[i] += 1
        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
        [t.start() for t in th]; [t.join() for t in th]
        dt = time.perf_counter() - t0
        samples.append(sum(done) / dt)
    return {"value": max(samples), "unit": "queries/s", "cores": cores, "kind": "port", "samples": samples,
            "sample": f"2 x {seconds / 2:.0f}s, cycling the {len(qk)} C3 queries on the full {a.bm25_docs}-doc index, {cores} pinned threads (one query each); "
                      "CPU restatement of the reference algorithms (no Rust toolchain here), not the reference binary"}


# ----------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of this run, written straight to the process's original stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    global _REAL_STDOUT, _OUTPUTS
    a = parse()
    # stdout carries exactly one JSON line: everything else any library writes to fd 1 (NCCL prints its version banner
    # there whenever NCCL_DEBUG >= VERSION) is sent to stderr instead
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    sections = [s for s in a.sections.split(",") if s]
    if a.impl == "reference":
        rank = int(os.environ.get("RANK", 0))
        if rank != 0:
            return 0
        import __graft_entry__ as g
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
        base = cpu_vector_baseline(a, max(a.cpu_seconds, 2.0) * max(1, min(a.steps, 3)))   # two pinned samples inside
        line = {"impl": "reference", "metric": "queries/sec at top-10 (1M x 768 f32 cosine brute-force kNN)", "value": base["value"],
                "unit": "queries/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": None,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"C2 brute-force cosine kNN: {a.rows} x {a.dims} f32, top-{TOPK} (restated reference CPU path, {base['cores']} threads)"},
                "cpu_baseline": base, "kind_note": "CPU restatement (port) of the reference algorithms: the Rust reference cannot be built on this image",
                "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if "bm25" in sections:
            try:
                line["bm25"] = {"cpu_baseline": cpu_bm25_baseline(a, a.cpu_seconds)}
                line["bm25"]["value"] = line["bm25"]["cpu_baseline"]["value"]
            except Exception as e:  # pragma: no cover
                line["bm25"] = {"error": repr(e)}
        emit(line)
        return 0

    if not torch.cuda.is_available():
        emit({"error": "no CUDA device: bench.py measures the B200 path only (no CPU fallback)"})
        return 1
    import __graft_entry__ as g
    if not os.path.exists(g.LIB):
        g.build()
    rank, world = dist_setup(a.gpus)
    if a.dump_outputs and rank == 0:       # at N>1 every rank returns the merged global results: rank 0 writes them
        _OUTPUTS = {}
    # one explicit (non-default) stream for everything: library kernels, torch CUDA events and NCCL collectives
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    out = {"n_gpus": world, "steps": a.steps, "warmup": a.warmup, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "impl": "b200"}
    parity = {}
    want_parity = "parity" in sections and a.parity_queries > 0
    ix, q_host = bench_vector(a, rank, world, out)
    if want_parity:
        try:
            parity["vector"] = parity_vector(a, ix, q_host, rank, world)
        except Exception as e:  # pragma: no cover
            parity["vector"] = {"error": repr(e)}
    ix.close()
    del ix
    torch.cuda.empty_cache()
    if "int8" in sections:
        try:
            out["int8"] = bench_vector_int8(a, rank, world)
        except Exception as e:  # pragma: no cover
            out["int8"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        if world == 1 and isinstance(out.get("int8"), dict):
            try:
                out["int8"]["variants"] = bench_vector_int8_variants(a, rank, world)
            except Exception as e:  # pragma: no cover
                out["int8"]["variants"] = {"error": repr(e)}
            torch.cuda.empty_cache()
    if "hybrid" in sections:
        try:
            out["hybrid"] = bench_hybrid(a, rank, world)
        except Exception as e:  # pragma: no cover
            out["hybrid"] = {"error": repr(e)}
        torch.cuda.empty_cache()
    if "phrase" in sections and world == 1:
        try:
            out["phrase"] = bench_phrase(a, rank, world)
        except Exception as e:  # pragma: no cover
            out["phrase"] = {"error": repr(e)}
        torch.cuda.empty_cache()
    if "bm25" in sections:
        lex_ix = None
        try:
            want_c5 = "c5" in sections and a.c5_docs == a.bm25_docs
            out["bm25"], lex_ix = bench_bm25(a, rank, world, keep_index=True, vector_dims=C2_DIMS if want_c5 else 0)
            if want_parity:
                try:
                    parity["bm25"] = parity_bm25(a, lex_ix, rank, world)
                except Exception as e:  # pragma: no cover
                    parity["bm25"] = {"error": repr(e)}
            if want_c5:
                try:
                    out["c5"] = bench_c5(a, rank, world, lex_ix)
                except Exception as e:  # pragma: no cover
                    out["c5"] = {"error": repr(e)}
        except Exception as e:  # pragma: no cover
            out["bm25"] = {"error": repr(e)}
        if lex_ix is not None:
            lex_ix.close()
        torch.cuda.empty_cache()
    if want_parity and rank == 0:
        ok = [v for v in parity.values() if isinstance(v, dict) and "mismatches" in v]
        out["parity_check"] = {"n": sum(v["n"] for v in ok), "mismatches": sum(v["mismatches"] for v in ok), "n_gpus": world,
                               "what": "merged top-10 of the first queries of each path vs the CPU oracle (exhaustive), checked on rank 0 after the timed regions",
                               **parity}
    if rank == 0 and world == 1 and a.cpu_seconds > 0:
        try:
            out["cpu_baseline"] = cpu_vector_baseline(a, a.cpu_seconds)
        except Exception as e:  # pragma: no cover
            out["cpu_baseline"] = {"error": repr(e)}
        if "int8" in sections and isinstance(out.get("int8"), dict) and "error" not in out["int8"]:
            try:
                out["int8"]["cpu_baseline"] = cpu_vector_int8_baseline(a, min(a.cpu_seconds, 8.0))
            except Exception as e:  # pragma: no cover
                out["int8"]["cpu_baseline"] = {"error": repr(e)}
        if "bm25" in sections and isinstance(out.get("bm25"), dict) and "error" not in out["bm25"]:
            try:
                out["bm25"]["cpu_baseline"] = cpu_bm25_baseline(a, a.cpu_seconds)
            except Exception as e:  # pragma: no cover
                out["bm25"]["cpu_baseline"] = {"error": repr(e)}
    if _OUTPUTS is not None:
        write_outputs(a.dump_outputs)
    if rank == 0:
        emit(out)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
