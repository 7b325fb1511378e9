#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on synthetic Llama-70B-shape matrices.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the workload `w4a16_gemv_llama70b`: the W4A16 (uint4, group 128, GPTQ-style
quantized zeros, interleaved storage) GEMV at M=1 for the Llama-2-70B linear shapes BASELINE.json configs[1] names
((N,K) = (8192,8192), (28672,8192), (8192,28672)) plus the target shape (12288,12288).  `value` = algorithmic bytes of
the step / device time (GB/s), inputs resident in HBM.  Before anything is timed, one shape is built from REAL quantised
fields through the product's own weight transform and a slice of its output is checked against the CPU oracle (a kernel
that is wrong at scale must not post a number).  The compute-bound half of the metric (W4A16 GEMM, M in {16,128,4096} on
the three Llama (N,K) pairs + M=4096 N=K=12288, TFLOPS) and the W2A8 path are measured in the same run and reported under
"gemm" / "gemm_llama" / "w2a8" with their own roofline objects.  `e2e` goes through the public operator API with HOST
activations (pinned H2D copy + D2H of the result inside the timed region, synchronised every step).  With --gpus N>1
(launched under torchrun) the weights are sharded along N across ranks (column parallel) and the outputs gathered:
strong scaling, max-over-ranks device time.

--impl reference times the reference's only CPU implementation of this path -- the torch dequantise+matmul reference
program of its tests (testing/python/operators/test_general_matmul_ops_backend_tl.py:227-273), restated in
oracle/bitblas_oracle.py -- on the host cores, on a bounded row sample of the SAME four shapes.

--dump-outputs DIR writes the four [1, N] outputs of the last timed GEMV step as DIR/gemv_N<N>_K<K>.npy (float32, exact for
the fp16 results).  Every input is generated from fixed seeds, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GEMV_SHAPES = [(8192, 8192), (28672, 8192), (8192, 28672), (12288, 12288)]  # (N, K)
GROUP = 128
GEMM_SHAPE = (4096, 12288, 12288)  # (M, N, K)
LLAMA_NK = [(8192, 8192), (28672, 8192), (8192, 28672)]
# the workload both arms are run on; identical in both JSON lines (everything arm-specific lives under other keys)
CONFIG = {"workload": "w4a16_gemv_llama70b", "shapes_NK": GEMV_SHAPES, "M": 1, "A_dtype": "float16", "W_dtype": "uint4",
          "group_size": GROUP, "zeros_mode": "quantized"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained"), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


def profiled_traffic():
    """DRAM bytes per launch of the dominant kernels, from the committed ncu capture (profiles/r2_traffic.json, written by
    tools/ncu_traffic.py out of an `ncu --set full` report; keyed to the commit it was taken at).  None if absent."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def gemv_bytes(N, K, M=1, bits=4, g=GROUP, zeros="quantized", a_bytes=2, out_bytes=2):
    """algorithmic bytes, SURVEY.md §8(d): W + scale + zeros + A + C."""
    b = N * K * bits // 8 + N * (K // g) * 2
    if zeros != "none":
        b += (K // g) * N * bits // 8 if zeros == "quantized" else N * (K // g) * 2
    return b + M * K * a_bytes + M * N * out_bytes


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: torch dequantise + matmul on the host cores (oracle/, kind "port")
# ---------------------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """torch intra-op threads for the CPU legs: all host cores unless that is slower than fewer (containers with a CPU
    quota below os.cpu_count() make an over-subscribed pool orders of magnitude slower); the count used is reported."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    x = torch.randint(0, 16, (2048, 2048), dtype=torch.int32)
    best, best_t = 1, None
    for nt in sorted({1, 4, 16, 64, ncpu}):
        if nt > ncpu:
            continue
        torch.set_num_threads(nt)
        (x - x).sum()
        t0 = time.perf_counter()
        for _ in range(3):
            (x - x).to(torch.float16)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    return best


class CpuWorkload:
    """The reference's CPU computation of the workload: for each of the four shapes a ROW SAMPLE (the first N/sample_div output
    features -- rows of W are independent dot products, so the GB/s of a row sample is the GB/s of the shape) of the
    un-packed int weight matrix, (w - z) * s in fp16, fp32 matmul (test_general_matmul_ops_backend_tl.py:227-273)."""

    def __init__(self, sample_div=16, cores=None):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import bitblas_oracle as O
        self.O = O
        self.cores = cores or pick_cpu_threads()
        torch.set_num_threads(self.cores)
        self.sample_div = sample_div
        g = torch.Generator().manual_seed(0)
        self.cases = []
        self.bytes = 0
        for N, K in GEMV_SHAPES:
            n = max(16, N // sample_div)
            fields = torch.randint(0, 16, (n, K), generator=g, dtype=torch.int32)
            scale = (torch.rand((n, K // GROUP), generator=g) * 0.1 + 0.01).half()
            zq = torch.randint(0, 16, (K // GROUP, n), generator=g, dtype=torch.int8)
            qz = torch.from_numpy(O.general_compress(zq.numpy(), 4))
            A = (torch.rand((1, K), generator=g) - 0.5).half()
            self.cases.append((A, fields, scale, qz))
            self.bytes += gemv_bytes(n, K)

    def step(self):
        O = self.O
        for A, fields, scale, qz in self.cases:
            O.matmul_dequant(A, fields, W_dtype="uint4", group_size=GROUP, with_scaling=True, with_zeros=True,
                             zeros_mode="quantized", scale=scale, zeros=qz)

    def matmul_fp16_only_ms(self):
        """context: the north star's "torch.matmul FP16 CPU path" alone, on pre-dequantised fp16 weights (same row sample)."""
        O = self.O
        ws = [(A, O.dequantize_weight(f, W_dtype="uint4", group_size=GROUP, with_scaling=True, with_zeros=True,
                                      zeros_mode="quantized", scale=s, zeros=z)) for A, f, s, z in self.cases]
        for A, Wd in ws:
            torch.matmul(A, Wd.T)
        ts = []
        for _ in range(10):   # BASELINE.md §3: 10 timed reps, median
            t0 = time.perf_counter()
            for A, Wd in ws:
                torch.matmul(A, Wd.T)
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts) * 1e3

    def describe(self, ms):
        return (f"row sample 1/{self.sample_div} of each of the 4 shapes {GEMV_SHAPES} (M=1, g={GROUP}, quantized zeros): torch "
                f"(w-z)*s in fp16 + fp32 matmul on the int weight matrix, {ms:.1f} ms per sampled pass, {self.cores} threads")


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    wl = CpuWorkload()
    for _ in range(max(1, min(args.warmup, 3))):
        wl.step()
    ts = []
    for _ in range(max(1, args.steps)):
        t0 = time.perf_counter()
        wl.step()
        ts.append(time.perf_counter() - t0)
    t = sum(ts) / len(ts)
    value = wl.bytes / t / 1e9
    sample = wl.describe(t * 1e3)
    line = {"metric": "w4a16_gemv_gbps_llama70b", "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic", "impl": "reference", "config": CONFIG,
            "cpu_baseline": {"value": value, "unit": "GB/s", "cores": wl.cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def make_linear(bitblas, N_local, K, dev, *, a_dtype="float16", w_dtype="uint4", zeros_mode="quantized", seed=0, M=(1, 4096)):
    """operator + random parameters generated directly in storage form on the device (any byte pattern is a valid
    packed uint4 pair, so no host transform is needed at 70B sizes)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    int_path = a_dtype == "int8"
    cfg = bitblas.MatmulConfig(M=list(M), N=N_local, K=K, A_dtype=a_dtype, W_dtype=w_dtype,
                               accum_dtype="int32" if int_path else "float16", out_dtype="int32" if int_path else "float16",
                               group_size=-1 if int_path else GROUP, with_scaling=not int_path, with_zeros=not int_path,
                               zeros_mode=zeros_mode)
    op = bitblas.Matmul(cfg, enable_tuning=False)
    wshape = op.retrieve_weight_shape()
    W = torch.randint(-128, 128, wshape, generator=g, dtype=torch.int8, device=dev)
    if int_path:
        return op, dict(W=W, scale=None, zeros=None)
    G = K // GROUP
    scale = (torch.rand((N_local, G), generator=g, device=dev) * 0.02 + 0.002).half()
    if zeros_mode == "quantized":
        zeros = torch.randint(-128, 128, (G, N_local // 2), generator=g, dtype=torch.int8, device=dev)
    else:
        zeros = torch.randint(0, 16, (N_local, G), generator=g, device=dev).half()
    return op, dict(W=W, scale=scale, zeros=zeros)


def oracle_gate(bitblas, dev):
    """Correctness gate, run before any timing: W4A16 at a BASELINE shape built from real quantised fields through the product's
    own device weight transform; M = 1 (the streaming kernel) and M = 16 (the tcgen05 kernel); 512 output features compared with
    the CPU oracle (rtol = atol = 1e-2 like the reference's tests).  Raises on mismatch."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import bitblas_oracle as O
    N, K, ncheck = 8192, 8192, 512
    g = torch.Generator().manual_seed(123)
    fields = torch.randint(0, 16, (N, K), generator=g, dtype=torch.int8)
    scale = (torch.rand((N, K // GROUP), generator=g) * 0.1 + 0.01).half()
    zq = torch.randint(0, 16, (K // GROUP, N), generator=g, dtype=torch.int8)
    qz = torch.from_numpy(O.general_compress(zq.numpy(), 4))
    cfg = bitblas.MatmulConfig(M=[1, 16], N=N, K=K, A_dtype="float16", W_dtype="uint4", accum_dtype="float16", out_dtype="float16",
                               group_size=GROUP, with_scaling=True, with_zeros=True, zeros_mode="quantized")
    op = bitblas.Matmul(cfg, enable_tuning=False)
    W = op.transform_weight(fields.to(dev))
    sc, zz = scale.to(dev), qz.to(dev)
    report = {}
    for m in (1, 16):
        A = (torch.rand((m, K), generator=g) - 0.5).half()
        got = op.forward(A.to(dev), W, scale=sc, zeros=zz).cpu()
        # the last `ncheck` output features (rows of W): scale rows and the matching packed-zero columns
        ref = O.matmul_dequant(A, fields[N - ncheck:].to(torch.int32), W_dtype="uint4", group_size=GROUP, with_scaling=True,
                               with_zeros=True, zeros_mode="quantized", scale=scale[N - ncheck:],
                               zeros=torch.from_numpy(O.general_compress(zq[:, N - ncheck:].numpy(), 4)))
        err = O.rel_fro_error(got[:, N - ncheck:], ref)
        O.torch_assert_close(got[:, N - ncheck:].float(), ref.float(), rtol=1e-2, atol=1e-2 * max(1.0, float(ref.float().abs().mean())),
                             max_mismatched_ratio=0.0)
        if not (err <= 1e-2):
            raise AssertionError(f"oracle gate failed: m={m} normwise rel err {err}")
        report[f"m{m}"] = {"kernel": op.kernel_for(m), "rel_fro_err": float(f"{err:.3e}")}
    return {"shape_NK": [N, K], "features_checked": ncheck, "criterion": "normwise <= 1e-2 and elementwise rtol=atol=1e-2, 0 mismatches", **report}


def dump_outputs(dirname, arrays, limit=64 << 20):
    """each tensor as <dirname>/<name>.npy in float32"""
    import numpy as np
    host = {name: t.float().cpu().numpy() for name, t in arrays.items()}
    assert sum(a.nbytes for a in host.values()) <= limit, "outputs to dump exceed 64 MB"
    os.makedirs(dirname, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def timed(fn, steps, warmup, barrier=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    return s.elapsed_time(e) / steps  # ms per step


def rotating_kernel_time(op, prm, A, out, reps=5, min_bytes=300 * 1024 * 1024):
    """per-launch kernel time with a cold L2: back-to-back launches cycling through enough read-only copies of the parameters
    that the working set (> 2x the 126 MB L2) can never be resident; median of `reps` passes.  The pass is captured in a CUDA
    graph (the launches keep their programmatic-dependent-launch edges) so that a ~10 us kernel is not timed against the ~10 us
    Python call that launches it; if capture is unavailable the launches are issued directly.  (No write-flush: dirty lines
    left in L2 by a flush kernel are written back DURING the timed kernel and charged to it -- measured +10..25 us.)"""
    wbytes = prm["W"].numel()
    ncopies = max(2, -(-min_bytes // wbytes))
    copies = [prm] + [{k: (v.clone() if v is not None else None) for k, v in prm.items()} for _ in range(ncopies - 1)]
    for c in copies:
        op.forward(A, c["W"], scale=c["scale"], zeros=c["zeros"], output=out)
    torch.cuda.synchronize()

    npass = max(2 * ncopies, 40)     # launches per pass: the graph-launch latency of a pass (a few us) is spread over >= 40 kernels

    def one_pass():
        for i in range(npass):
            c = copies[i % ncopies]
            op.forward(A, c["W"], scale=c["scale"], zeros=c["zeros"], output=out)

    graph = None
    if os.environ.get("BB_BENCH_GRAPH", "1") != "0":
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                one_pass()                      # warm-up on the capture stream (workspace for this stream, attributes)
                side.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    one_pass()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
        except Exception as ex:  # noqa: BLE001
            print(f"[bench] CUDA graph capture unavailable ({ex}); timing direct launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        if graph is not None:
            graph.replay()
        else:
            one_pass()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) / npass)
    return statistics.median(ts), ncopies, graph is not None


def int8_peak_tops(dev):
    """dense int8 tensor-core throughput of this GPU through cuBLASLt (torch._int_mm, 8192^3), burst: the denominator of the
    W2A8 GEMM fraction (MEASURED_PEAKS.json has no int8 entry)."""
    try:
        a = torch.randint(-128, 128, (8192, 8192), dtype=torch.int8, device=dev)
        b = torch.randint(-128, 128, (8192, 8192), dtype=torch.int8, device=dev).t()
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = None
        for _ in range(10):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            torch._int_mm(a, b)
            e.record()
            torch.cuda.synchronize()
            t = s.elapsed_time(e)
            best = t if best is None or t < best else best
        return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--only", default="", help="comma list of sections to run: gemm,llama,w2a8,formats,e2e (default all; the GEMV step always runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed GEMV step as DIR/<name>.npy (float32; single GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    rank, world, local = dist_env()
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs needs a single-GPU run")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    import bitblas_b200 as bitblas
    from bitblas_b200 import _lib
    lib = _lib.load()
    pk = peaks()
    traffic = profiled_traffic()
    only = set(x for x in args.only.split(",") if x)
    want = lambda s: not only or s in only  # noqa: E731
    warmup = max(3, args.warmup)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather(out_local, m):
        """column-parallel exchange step, NCCL flavour: all-gather of [m, N/G] partial outputs (bitblas_b200/parallel.py)."""
        if world == 1:
            return out_local
        g = torch.empty((world * m, out_local.shape[-1]), dtype=out_local.dtype, device=dev)
        dist.all_gather_into_tensor(g, out_local)
        return g

    # ---- correctness gate (rank 0 checks; every rank must pass before anything is timed) ----
    gate = oracle_gate(bitblas, dev)

    # fused flavour: the kernel epilogue stores this rank's column slice into every rank's output (symmetric memory over
    # NVLink), then one device-side barrier -- no separate collective (bb_matmul_scatter)
    fused = {"on": False}
    symm_cache = {}
    peer_arrays = {}   # id(symmetric-memory handle) -> prebuilt (c_void_p * world) array of the peers' buffer pointers
    if world > 1 and os.environ.get("BB_BENCH_FUSED", "1") != "0":
        try:
            import torch.distributed._symmetric_memory as symm_mem

            def symm_out(m, N, dtype, tag=None):
                key = (m, N, dtype, tag)
                if key not in symm_cache:
                    pairs = []
                    for _ in range(2):
                        t = symm_mem.empty((m, N), dtype=dtype, device=dev)
                        h = symm_mem.rendezvous(t, dist.group.WORLD)
                        ptrs = [int(p) for p in h.buffer_ptrs]
                        peer_arrays[id(h)] = (ctypes.c_void_p * len(ptrs))(*[ctypes.c_void_p(p) for p in ptrs])  # built once
                        pairs.append((t, h))
                    symm_cache[key] = [pairs, 0]
                e = symm_cache[key]
                t, h = e[0][e[1]]
                e[1] ^= 1
                return t, h

            t_, h_ = symm_out(1, 16 * world, torch.float16)
            h_.barrier(channel=0)
            torch.cuda.synchronize()
            fused["on"] = True
            if os.environ.get("BB_BENCH_PEER_BARRIER", "1") != "0":
                from bitblas_b200.parallel import PeerBarrier
                fused["barrier"] = PeerBarrier(dev)      # bb_peer_barrier: the library's own one-kernel barrier
        except Exception as ex:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] symmetric memory unavailable ({ex}); using NCCL all-gather", file=sys.stderr)

    def run_sharded(op, prm, A, out_local, m, N_full, defer=None):
        """one column-parallel matmul: returns the full [m, N] output tensor of this rank.  `defer` (a list): do not barrier
        here -- the caller issues ONE device barrier for all the projections of the step (their results become visible on every
        rank together); the buffer tag keeps projections with equal N apart."""
        if world == 1:
            op.forward(A, prm["W"], scale=prm["scale"], zeros=prm["zeros"], output=out_local)
            return out_local
        if fused["on"]:
            buf, hdl = symm_out(m, N_full, out_local.dtype, tag=id(op))
            op.forward_scatter(A, prm["W"], scale=prm["scale"], zeros=prm["zeros"],
                               peer_ptrs=peer_arrays.get(id(hdl)) or [int(p) for p in hdl.buffer_ptrs],
                               ldc=N_full, col_offset=rank * (N_full // world))
            if defer is not None:
                defer.append(hdl)
            elif fused.get("barrier") is not None:
                fused["barrier"]()
            else:
                hdl.barrier(channel=0)
            return buf
        op.forward(A, prm["W"], scale=prm["scale"], zeros=prm["zeros"], output=out_local)
        return gather(out_local, m)

    result = {"oracle_gate": gate}
    sampler = ClockSampler(torch.cuda.current_device())
    # ---------------- GEMV (the headline workload) ----------------
    # Every step streams parameters that cannot be L2-resident: at world = 1 the step's own 357 MB exceed the 126 MB L2; with the
    # weights sharded over `world` GPUs the per-GPU share shrinks below it, so the step cycles through `nsets` independent
    # parameter sets (>= 300 MB per GPU in total) -- step i uses set i % nsets.
    total_bytes = sum(gemv_bytes(N, K) for N, K in GEMV_SHAPES)
    per_gpu = sum(gemv_bytes(N // world, K) for N, K in GEMV_SHAPES)
    nsets = 1 if per_gpu > 300e6 else -(-int(300e6) // per_gpu)
    if world > 1 and nsets % 2:
        nsets += 1                # the fused path alternates two symmetric output buffers per projection: keep the cycle even
    sets = []
    for c in range(nsets):
        ops_c = []
        for i, (N, K) in enumerate(GEMV_SHAPES):
            if c == 0:
                op, prm = make_linear(bitblas, N // world, K, dev, seed=i)
                A = (torch.rand((1, K), generator=torch.Generator(device=dev).manual_seed(100 + i), device=dev) - 0.5).half()
                out = torch.empty((1, N // world), dtype=torch.float16, device=dev)
            else:
                op, prm0, A, out = sets[0][i][:4]
                prm = {k: (v.clone() if v is not None else None) for k, v in prm0.items()}
            ops_c.append((op, prm, A, out, N, K))
        sets.append(ops_c)
    ops = sets[0]

    step_sync = os.environ.get("BB_BENCH_STEP_BARRIER", "1") != "0"   # one device barrier per step instead of per projection

    def gemv_step_on(ops_c):
        pending = [] if (world > 1 and fused["on"] and step_sync) else None
        for op, prm, A, out, N, K in ops_c:
            run_sharded(op, prm, A, out, 1, N, defer=pending)
        if pending:   # peer stores of all four projections precede the barrier in stream order on every rank
            if fused.get("barrier") is not None:
                fused["barrier"]()
            else:
                pending[-1].barrier(channel=0)

    # The step is captured once per parameter set in a CUDA graph (four launches with their programmatic-dependent-launch
    # edges + the device barrier) and replayed: at 8 GPUs a shard's kernel takes a few microseconds, the four Python calls that
    # launch them do not.  Same code path at every world size; BB_BENCH_STEP_GRAPH=0 (or a failed capture) issues the launches directly.
    step_graphs, launches_per_step, step_block = None, None, None
    if os.environ.get("BB_BENCH_STEP_GRAPH", "1") != "0":
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            gs = []
            with torch.cuda.stream(side):
                for ops_c in sets:                  # warm-up on the capture stream: per-stream workspaces, symmetric buffers
                    gemv_step_on(ops_c)
                side.synchronize()
                barrier()
                for ops_c in sets:
                    l0 = lib.bb_launch_count()
                    gph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gph, stream=side):
                        gemv_step_on(ops_c)
                    launches_per_step = lib.bb_launch_count() - l0
                    gs.append(gph)
                # a block of consecutive steps in ONE graph (a decoder runs its layers' projections back to back: the launch-bound
                # inner loop belongs in one graph); the remainder of --steps is replayed step by step
                block_len = nsets * max(1, round(10 / nsets))
                block = torch.cuda.CUDAGraph()
                with torch.cuda.graph(block, stream=side):
                    for j in range(block_len):
                        gemv_step_on(sets[j % nsets])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            step_graphs = gs
            step_block = (block, block_len)
        except Exception as ex:  # noqa: BLE001
            print(f"[bench] step graph capture unavailable on rank {rank} ({ex}); issuing launches directly", file=sys.stderr)
            step_graphs, step_block = None, None
            torch.cuda.synchronize()
    if world > 1:   # the choice must be collective: a rank replaying a graph and a rank launching directly still meet in the barrier, but keep it simple
        flag = torch.tensor([1 if step_graphs is not None else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            step_graphs, step_block = None, None
    step_no = [0]

    def gemv_step():
        c = step_no[0] % nsets
        step_no[0] += 1
        if step_graphs is not None:
            step_graphs[c].replay()
        else:
            gemv_step_on(sets[c])

    if rank == 0:
        sampler.start()
    def run_steps(k):
        """exactly k steps: whole blocks (one graph launch per `block_len` steps), then the remainder one step per graph launch"""
        if step_block is not None:
            nb, rem = divmod(k, step_block[1])
            for _ in range(nb):
                step_block[0].replay()
            step_no[0] = 0          # the remainder continues the parameter-set rotation where a block ends
        else:
            rem = k
        for _ in range(rem):
            gemv_step()

    run_steps(warmup)
    if step_block is not None:
        step_block[0].replay()      # (the block graph itself, whatever --warmup is)
    torch.cuda.synchronize()
    launches0 = lib.bb_launch_count()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    run_steps(args.steps)
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    ms_step = ev0.elapsed_time(ev1) / args.steps
    if args.dump_outputs:   # every parameter set writes the same `out` tensors: they hold the last timed step's results
        dump_outputs(args.dump_outputs, {f"gemv_N{N}_K{K}": out for op, prm, A, out, N, K in ops})
    # kernels of this library launched inside the timed region (replayed graph launches are not seen by the library's counter)
    launches = (launches_per_step * args.steps) if step_graphs is not None else (lib.bb_launch_count() - launches0)
    ms_step = max_over_ranks(ms_step)
    value = total_bytes / (ms_step * 1e-3) / 1e9
    result["step_method"] = {"cuda_graph": step_graphs is not None, "steps_per_graph_launch": step_block[1] if step_block else 1,
                             "parameter_sets": nsets,
                             "per_gpu_bytes_per_step": per_gpu}

    # per-shape kernel time, cold L2 (rotating parameter copies)
    per_shape = []
    for op, prm, A, out, N, K in ops:
        t, ncopies, graphed = rotating_kernel_time(op, prm, A, out)
        b = gemv_bytes(N // world, K)
        per_shape.append({"N": N, "K": K, "us": round(t * 1e3, 2), "GBps": round(b / (t * 1e-3) / 1e9, 1),
                          "frac_hbm": round(b / (t * 1e-3) / 1e9 / pk["hbm"], 3), "kernel": op.kernel_for(1), "copies": ncopies,
                          "cuda_graph": graphed})
    tgt = per_shape[-1]
    tr = traffic.get("gemv_m1_12288") if world == 1 else None
    roofline = {"bound": "hbm", "kernel": f"{tgt['kernel']} (W4A16 m=1 N=K=12288)", "achieved": tgt["GBps"],
                "peak": pk["hbm"], "unit": "GB/s", "frac": tgt["frac_hbm"],
                "traffic": tr.get("dram_bytes") if tr else None, "traffic_source": tr.get("source") if tr else None,
                "algorithmic_bytes": gemv_bytes(12288 // world, 12288), "us": tgt["us"], "peak_source": pk["src"],
                "timing": "CUDA events around back-to-back launches (one CUDA graph per pass) cycling through >= 300 MB of read-only parameter copies (cold L2), per-launch average, median of 5"}
    result["gemv_shapes"] = per_shape

    def gemm_point(op, prm, m, N, K, reps):
        A = (torch.rand((m, K), device=dev) - 0.5).half()
        out = torch.empty((m, N // world), dtype=torch.float16, device=dev)
        ms = max_over_ranks(timed(lambda: run_sharded(op, prm, A, out, m, N), reps, 3, barrier))
        tf = 2.0 * m * N * K / (ms * 1e-3) / 1e12
        b = gemv_bytes(N, K, M=m)
        t_mem, t_fl = b / (pk["hbm"] * 1e9), 2.0 * m * N * K / (pk["tf"] * 1e12)
        return {"M": m, "N": N, "K": K, "us": round(ms * 1e3, 2), "TFLOPS": round(tf, 1), "GBps": round(b / (ms * 1e-3) / 1e9, 1),
                "frac_tensor": round(tf / pk["tf"], 3), "frac_of_max_roofline": round(max(t_mem, t_fl) / (ms * 1e-3), 3),
                "kernel": op.kernel_for(m)}

    # ---------------- GEMM M=4096 N=K=12288 (tensor-bound half of the metric) + small M ----------------
    if want("gemm"):
        M, N, K = GEMM_SHAPE
        op, prm = make_linear(bitblas, N // world, K, dev, seed=11)
        g4 = gemm_point(op, prm, M, N, K, 10)
        trg = traffic.get("gemm_m4096_12288") if world == 1 else None
        result["gemm"] = {"M": M, "N": N, "K": K, "ms": round(g4["us"] / 1e3, 4), "TFLOPS": g4["TFLOPS"], "kernel": g4["kernel"],
                          "roofline": {"bound": "tensor", "achieved": g4["TFLOPS"], "peak": pk["tf"], "unit": "TFLOP/s",
                                       "frac": g4["frac_tensor"],
                                       "frac_of_sustained": round(g4["TFLOPS"] / pk["tf_sustained"], 3) if pk["tf_sustained"] else None,
                                       "traffic": trg.get("dram_bytes") if trg else None, "traffic_source": trg.get("source") if trg else None,
                                       "algorithmic_flops": 2.0 * M * N * K, "peak_source": pk["src"],
                                       "note": "A (100 MB) + W (75 MB) exceed L2; 10 back-to-back launches"}}
        result["gemm_small_m"] = [gemm_point(op, prm, m, N, K, 20) for m in (16, 128)]
        del op, prm

    # ---------------- BASELINE configs[2]: W4A16 GEMM M in {16,128,4096} on the three Llama-70B (N,K) pairs ----------------
    if want("llama"):
        rows = []
        for i, (N, K) in enumerate(LLAMA_NK):
            op, prm = make_linear(bitblas, N // world, K, dev, seed=30 + i)
            for m in (16, 128, 4096):
                rows.append(gemm_point(op, prm, m, N, K, 10 if m == 4096 else 20))
            del op, prm
        result["gemm_llama"] = rows

    # ---------------- W2A8 (BitNet), same cold-L2 method as W4A16 ----------------
    if want("w2a8"):
        N, K = 12288, 12288
        op8, prm8 = make_linear(bitblas, N // world, K, dev, a_dtype="int8", w_dtype="int2", seed=21, M=(1, 128))
        i8peak = int8_peak_tops(dev) if world == 1 else None
        w2 = []
        for m in (1, 128):
            A8 = torch.randint(-128, 128, (m, K), dtype=torch.int8, device=dev)
            out8 = torch.empty((m, N // world), dtype=torch.int32, device=dev)
            if world == 1:
                t8, _, _ = rotating_kernel_time(op8, prm8, A8, out8)
            else:
                t8 = max_over_ranks(timed(lambda: run_sharded(op8, prm8, A8, out8, m, N), 20, 3, barrier))
            b = N * K // 4 + m * K + m * N * 4
            tops = 2.0 * m * N * K / (t8 * 1e-3) / 1e12
            row = {"M": m, "us": round(t8 * 1e3, 2), "GBps": round(b / (t8 * 1e-3) / 1e9, 1), "TOPS": round(tops, 1),
                   "frac_hbm": round(b / (t8 * 1e-3) / 1e9 / pk["hbm"], 3), "kernel": op8.kernel_for(m)}
            if i8peak:
                row["frac_int8_peak"] = round(tops / i8peak, 4)
            w2.append(row)
        result["w2a8"] = w2
        result["int8_peak_tops_measured"] = round(i8peak, 1) if i8peak else None

    # ---------------- table formats (NF4) on the fast kernels: decode GEMV and tcgen05 GEMM at the target shape ----------------
    if want("formats") and world == 1:
        N, K = 12288, 12288
        cfgn = bitblas.MatmulConfig(M=[1, 4096], N=N, K=K, A_dtype="float16", W_dtype="nf4", accum_dtype="float16", out_dtype="float16",
                                    group_size=GROUP, with_scaling=True, with_zeros=False)
        opn = bitblas.Matmul(cfgn, enable_tuning=False)
        gn = torch.Generator(device=dev).manual_seed(5)
        prmn = dict(W=torch.randint(-128, 128, opn.retrieve_weight_shape(), generator=gn, dtype=torch.int8, device=dev),
                    scale=(torch.rand((N, K // GROUP), generator=gn, device=dev) * 0.02 + 0.002).half(), zeros=None)
        An = (torch.rand((1, K), device=dev) - 0.5).half()
        outn = torch.empty((1, N), dtype=torch.float16, device=dev)
        tn, _, _ = rotating_kernel_time(opn, prmn, An, outn)
        bn = gemv_bytes(N, K, zeros="none")
        rowsn = [{"W_dtype": "nf4", "M": 1, "us": round(tn * 1e3, 2), "GBps": round(bn / (tn * 1e-3) / 1e9, 1),
                  "frac_hbm": round(bn / (tn * 1e-3) / 1e9 / pk["hbm"], 3), "kernel": opn.kernel_for(1)}]
        A4 = (torch.rand((4096, K), device=dev) - 0.5).half()
        out4 = torch.empty((4096, N), dtype=torch.float16, device=dev)
        ms4 = timed(lambda: opn.forward(A4, prmn["W"], scale=prmn["scale"], output=out4), 10, 3)
        tf4 = 2.0 * 4096 * N * K / (ms4 * 1e-3) / 1e12
        rowsn.append({"W_dtype": "nf4", "M": 4096, "us": round(ms4 * 1e3, 1), "TFLOPS": round(tf4, 1), "frac_tensor": round(tf4 / pk["tf"], 3),
                      "kernel": opn.kernel_for(4096)})
        result["table_formats"] = rowsn
        del opn, prmn, A4, out4

    # ---------------- e2e: public API, host activations in, host results out, one sync per step ----------------
    e2e = None
    if want("e2e"):
        # one pinned staging buffer for the step's four activation vectors and one for its four results: the host issues ONE H2D
        # copy, the four Matmul.forward calls on views of the device buffer, and ONE D2H copy per step
        Ks, Ns = [K for _, K in GEMV_SHAPES], [N for N, _ in GEMV_SHAPES]
        hostA = torch.empty((sum(Ks),), dtype=torch.float16).pin_memory().copy_(torch.rand(sum(Ks)) - 0.5)
        hostC = torch.empty((sum(Ns),), dtype=torch.float16).pin_memory()
        devA = torch.empty((sum(Ks),), dtype=torch.float16, device=dev)
        devC = torch.empty((sum(Ns),), dtype=torch.float16, device=dev)
        a_views, c_views, ka, na = [], [], 0, 0
        for N, K in GEMV_SHAPES:
            a_views.append(devA[ka:ka + K].view(1, K)); ka += K
            c_views.append(devC[na:na + N].view(1, N)); na += N
        stream = torch.cuda.current_stream()

        e2e_no = [0]

        def e2e_step():
            devA.copy_(hostA, non_blocking=True)
            ops_c = sets[e2e_no[0] % nsets]      # same cold-L2 rotation as the device-timed step
            e2e_no[0] += 1
            for (op, prm, A, out, N, K), av, cv in zip(ops_c, a_views, c_views):
                if world == 1:
                    op.forward(av, prm["W"], scale=prm["scale"], zeros=prm["zeros"], output=cv)
                else:
                    cv.copy_(run_sharded(op, prm, av, out, 1, N).reshape(1, -1))
            hostC.copy_(devC, non_blocking=True)
            stream.synchronize()   # one host-visible result per step: all four projections' outputs are in pinned memory here

        ms_eager = max_over_ranks(timed(e2e_step, args.steps, warmup, barrier))
        ms_e, how, ms_graph = ms_eager, "eager: one Python call per projection", None
        # the package's own step capture (bitblas_b200.CapturedStep): the same copies and the same four forwards as ONE CUDA graph;
        # the host still writes the pinned input, launches, synchronises and reads the pinned output every step
        if world == 1 and os.environ.get("BB_BENCH_E2E_GRAPH", "1") != "0":
            try:
                def four():
                    for (op, prm, A, out, N, K), av, cv in zip(ops, a_views, c_views):
                        op.forward(av, prm["W"], scale=prm["scale"], zeros=prm["zeros"], output=cv)
                cap = bitblas.CapturedStep(four, h2d=[(devA, hostA)], d2h=[(hostC, devC)])
                for _ in range(warmup):
                    cap()
                torch.cuda.synchronize()
                t0 = time.perf_counter()            # every step ends in a host synchronise: wall clock IS the end-to-end time
                for _ in range(args.steps):
                    cap()                            # replay + stream synchronise
                ms_g = (time.perf_counter() - t0) * 1e3 / args.steps
                ms_graph = ms_g
                if ms_g < ms_e:
                    ms_e, how = ms_g, "bitblas_b200.CapturedStep: H2D + 4 x Matmul.forward + D2H replayed as one CUDA graph, synchronised every step"
            except Exception as ex:  # noqa: BLE001
                print(f"[bench] CapturedStep unavailable ({ex}); e2e is the eager path", file=sys.stderr)
        e2e = {"value": round(total_bytes / (ms_e * 1e-3) / 1e9, 1), "unit": "GB/s", "ms_per_step": round(ms_e, 4),
               "h2d_bytes_per_step": sum(K * 2 for _, K in GEMV_SHAPES), "d2h_bytes_per_step": sum(N * 2 for N, _ in GEMV_SHAPES),
               "path": how, "eager_ms_per_step": round(ms_eager, 4), "captured_step_ms_per_step": round(ms_graph, 4) if ms_graph else None,
               "note": "per step: ONE pinned H2D copy of the four activation vectors, 4 x Matmul.forward on views of it, ONE D2H copy of the four outputs into pinned memory, then ONE stream synchronise -- the host reads the step's results after it"}

    clocks = sampler.stop() if rank == 0 else None
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        wl = CpuWorkload()
        wl.step()
        ts = []
        for _ in range(10):   # BASELINE.md §3: 3 warm-ups (1 here: ~0.5 s each), 10 timed reps, median
            t0 = time.perf_counter()
            wl.step()
            ts.append(time.perf_counter() - t0)
        t = statistics.median(ts)
        mm_ms = wl.matmul_fp16_only_ms()
        cpu = {"value": round(wl.bytes / t / 1e9, 4), "unit": "GB/s", "cores": wl.cores, "kind": "port", "sample": wl.describe(t * 1e3),
               "matmul_fp16_only_ms": round(mm_ms, 3),
               "matmul_fp16_only_note": "the north star's torch.matmul-FP16 CPU path on PRE-dequantised fp16 weights, same row sample"}
        # the two host-side ratios a reader wants next to the GPU number, on the same bytes: dequant+matmul and matmul only
        gpu_ms_equiv = ms_step / wl.sample_div
        result["vs_cpu"] = {"dequant_matmul_ratio": round(t * 1e3 / gpu_ms_equiv, 1), "matmul_fp16_only_ratio": round(mm_ms / gpu_ms_equiv, 1),
                            "note": f"CPU time for a 1/{wl.sample_div} row sample of the step / (GPU step time / {wl.sample_div})"}

    if rank == 0:
        par = (f"column-parallel x{world}, " + (("fused peer-store epilogue over NVLink (bb_matmul_scatter) + one device barrier ("
               + ("bb_peer_barrier" if fused.get("barrier") is not None else "symmetric-memory library barrier") + ") per "
               + ("step" if step_sync else "projection")) if fused["on"] else "NCCL all-gather")) if world > 1 else "single GPU"
        line = {"metric": "w4a16_gemv_gbps_llama70b", "value": round(value, 1), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": CONFIG,
                "config_detail": {"parallelism": par,
                                  "l2": f"inputs larger than L2: each step streams {per_gpu / 1e6:.0f} MB per GPU and steps cycle through {nsets} independent parameter set(s) (>= 300 MB per GPU vs the 126 MB L2); per-shape numbers rotate >= 300 MB of parameter copies"},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}
        line.update(result)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
