#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config fwd|fwdbwd|cascade|train8]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W      (one rank per GPU)

--config fwd (default, BASELINE configs[1], the judged line): image-pairs/sec of the MaskFlownet-S forward at 1024x448,
batch 8 per GPU, synthetic uint8 pairs, random-init (MSRAPrelu) weights, replicas (no data-path collective).
One "step" = uint8 pairs -> /255 -> centralize -> 6-level forward -> Upsample(4) of the finest flow.  Arithmetic: fp32 in
and out; every contraction (correlations, deformable warp, all 3x3 / transposed convolutions) runs on OUR tensor-core
kernels with each operand split into bf16 hi + bf16 lo (hi*hi + hi*lo + lo*hi, fp32 accumulation: ~2^-17 relative, inside
the 1e-4 bound of north_star; no cuDNN / cuBLAS kernel runs in the step).
  value            device-resident inputs, the step replayed from a CUDA graph (network.FlowPredictor), K steps, CUDA events
  value_sustained  the same loop repeated until >= --sustain-seconds inside the same protocol (power-capped clocks)
  e2e              the public serving API (network.PipelinedFlowPredictor) with HOST buffers: pinned uint8 H2D and pinned
                   fp32 flow D2H inside the timed region, overlapped with the forward on copy streams
  roofline         level-2 correlation launch timed inside an eager step with CUDA events (+ every correlation and warp
                   launch; K3 against HBM bytes and bf16 flops); `traffic` = dram bytes per launch from the committed ncu
                   capture of the same kernel (static: ncu cannot run inside the timed region)
  cpu_baseline     oracle port of the whole forward on the host cores + the correlation-only table of BASELINE.md section 3
                   (1-thread literal MXNet loop nest / OpenMP all cores / torch-CPU) per pair, configs[0] first
--config fwdbwd  (configs[2])  MaskFlownet-S forward + MultiscaleEpe + backward, batch 8, 512x384 (3x3 convolutions: forward
                               on the tcgen05 kernel, backward cuDNN fp32 -- `--train-tc-forward 0` = cuDNN both ways;
                               MultiscaleEpe = the fused kernels of csrc/loss.cu)
--config cascade (configs[3])  MaskFlownet (S head + dual pyramid, md=2 correlations) forward, batch 4, 1024x448
--config train8  (configs[4])  training step, batch 4 per GPU (32 on 8 GPUs), 960x540 padded to 960x576 like
                               do_batch_mx (network/pipeline.py:122-130): fwd + bwd + ONE NCCL all-reduce + Adam

--impl reference times the CPU arm: the reference's own CPU path cannot run here (MXNet is not installable, SURVEY.md
section 8c), so it is the oracle port (oracle/network_ref.py: torch-CPU convolutions + the C oracle's OpenMP correlation /
deformable convolution) on the host threads, one image pair per step (a bounded sample of the same workload).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVEL_C = {6: 196, 5: 128, 4: 96, 3: 64, 2: 32}
ARITH = "f32 I/O; bf16 hi+lo split operands (hi*hi+hi*lo+lo*hi) on tensor cores, fp32 accumulate"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md 6.65 TB/s, 1.59 PFLOP/s)"


def dram_traffic(kernel_name: str):
    """dram read+write bytes per launch of the named kernel from the committed ncu captures (profiles/r0?_dram_traffic.json)."""
    for fn in ("r02_dram_traffic.json", "r01_dram_traffic.json"):
        try:
            for key, rec in json.load(open(os.path.join(ROOT, "profiles", fn))).items():
                if not key.startswith("_") and key in (kernel_name or ""):
                    return int(rec["dram_read_bytes"]) + int(rec["dram_write_bytes"]), f"static: profiles/{fn} (ncu --set full)"
        except (OSError, ValueError, KeyError):
            pass
    return None, "no ncu capture of this kernel committed"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.05)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=3)
        return self.summary()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        out = {"sm_mhz": mhz[len(mhz) // 2] if mhz else None,
               "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
               "reasons": reasons, "samples": len(self.samples)}
        try:
            out["power_w_max"] = max(float(s[6]) for s in self.samples if len(s) > 6)
        except ValueError:
            pass
        return out


def synthetic_pairs(n, seed, H, W):
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(0, 256, (n, 3, H, W), dtype=torch.uint8, generator=g)
    b = torch.randint(0, 256, (n, 3, H, W), dtype=torch.uint8, generator=g)
    return a, b


# ------------------------------------------------------------------------------------------------- CPU arm
def usable_host_threads() -> int:
    """Threads this process can actually run on: the affinity mask capped by the cgroup CPU quota (a GPU box exposes 128
    logical CPUs to a container that is allowed ~16 of them; running 128 OpenMP threads there measures oversubscription)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2: "<quota> <period>" or "max <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, per = int(f.read()), int(g.read())
                if q > 0:
                    n = min(n, max(1, (q + per // 2) // per))
        except (OSError, ValueError):
            pass
    return max(1, n)


def cpu_arm(steps: int, warmup: int, max_threads: int, H=448, W=1024):
    """Oracle port of the same forward on the host cores; one pair per step.  The thread count is the fastest of a short
    probe over {8, 16, 32, 64, all usable} (more threads only add contention on the small pyramid levels)."""
    from oracle import cref, network_ref
    from maskflownet_b200.network import MaskFlownetS
    model = MaskFlownetS()
    params = {k: v.detach() for k, v in model.named_parameters()}
    a, b = synthetic_pairs(1, 0, H, W)

    def run(n, threads):
        torch.set_num_threads(threads)
        cref.lib().mfn_ref_set_num_threads(threads)
        t0 = time.perf_counter()
        with torch.no_grad():
            for _ in range(n):
                network_ref.predict_flow(params, a, b, threads=threads)
        return (time.perf_counter() - t0) / n

    cands = sorted({t for t in (8, 16, 32, 64, max_threads) if t <= max_threads})
    probe = {t: run(1, t) for t in cands}
    best = min(probe, key=probe.get)
    for _ in range(max(0, warmup - 1)):
        run(1, best)
    sec = run(steps, best)
    return 1.0 / sec, sec, best


def cpu_corr_table(max_threads: int):
    """BASELINE.md section 3: the correlation alone on the host, per image pair (N = 1), ms per call:
    A = literal MXNet loop nest, 1 thread (MXNet's CPU operator has no OpenMP pragma); B = the same with OpenMP, best of
    {4, 16, all usable} threads; C = torch-CPU restatement (81 shifted multiply-means).  configs[0] (1,196,6,8) first, then cfg2 levels."""
    import numpy as np
    from oracle import cref, torch_ref
    rows = []
    shapes = [("cfg0_L6_384x512", (1, 196, 6, 8))] + [(f"cfg1_L{L}_448x1024", (1, LEVEL_C[L], 448 >> L, 1024 >> L))
                                                       for L in (6, 5, 4, 3, 2)]
    rng = np.random.default_rng(0)
    for name, shp in shapes:
        f1, f2 = rng.standard_normal(shp).astype(np.float32), rng.standard_normal(shp).astype(np.float32)

        def t_of(fn, reps):                 # best of reps: the host's most favourable number (libgomp team re-sizing
            fn()                            # makes the first calls at a new thread count erratic)
            best = float("inf")
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                best = min(best, time.perf_counter() - t0)
            return best * 1e3
        big = shp[1] * shp[2] * shp[3] > 200000
        a = t_of(lambda: cref.correlation_forward(f1, f2, threads=1), 2 if big else 5)
        bt = {t: t_of(lambda t=t: cref.correlation_forward(f1, f2, threads=t), 5 if big else 20)
              for t in sorted({min(4, max_threads), min(16, max_threads), max_threads})}
        tb = min(bt, key=bt.get)
        torch.set_num_threads(max_threads)
        t1, t2 = torch.from_numpy(f1), torch.from_numpy(f2)
        c = t_of(lambda: torch_ref.correlation(t1, t2, 4), 3 if big else 5)
        rows.append({"shape": name, "nchw": list(shp), "ms_1thread_literal": round(a, 3),
                     "ms_openmp_best": round(bt[tb], 3), "openmp_threads": tb, "ms_torch_cpu": round(c, 3)})
    return {"unit": "ms per call (best of reps), one image pair", "threads_usable": max_threads, "rows": rows}


# ------------------------------------------------------------------------------------------------- helpers
class Ctx:
    pass


def setup_gpu():
    from maskflownet_b200 import dist as mdist
    c = Ctx()
    c.rank, c.local, c.world = mdist.init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU implementation (use --impl reference for "
                         "the CPU arm)")
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    torch.backends.cudnn.allow_tf32 = False           # training-mode autograd convolutions stay fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    c.flush = torch.empty(256 << 20, dtype=torch.uint8, device=c.dev)
    c.mdist = mdist
    return c


def barrier(c):
    if c.world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


def timed(c, fn, K, sync_extra=None):
    """EXACTLY K calls of fn bracketed by barrier + synchronize; 256 MiB L2 flush before every call (inside the region);
    device time from CUDA events, max over ranks."""
    barrier(c)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        c.flush.zero_()
        fn()
    if sync_extra is not None:
        sync_extra()      # copy streams joined into the timed region (their work must finish before e1)
    e1.record()
    barrier(c)
    return c.mdist.max_over_ranks(e0.elapsed_time(e1), c.dev)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Write {name: float32 array} as <directory>/<name>.npy: what the timed path returned in its last step, for comparing
    two builds output for output (the inputs and weights are seeded, so equal arguments give equal inputs).  Compare with a
    tolerance: the centralize mean and the warp backward's input / weight gradients are atomic fp32 sums, and cuDNN picks
    its backward algorithms at run time, so repeated runs of one build differ in the last bits."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def base_line(metric, value, K, Wm, ms_total, world, config):
    return {"metric": metric, "value": round(value, 3), "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": round(ms_total / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config}


# ------------------------------------------------------------------------------------------------- configs[1]: forward
def bench_fwd(args, K, Wm):
    from maskflownet_b200 import _lib, network, ops
    c = setup_gpu()
    H, W, BATCH = 448, 1024, 8
    METRIC = "image-pairs/sec (MaskFlownet-S forward, 1024x448)"
    torch.manual_seed(0)
    model = network.MaskFlownetS().to(c.dev).eval()
    a_h, b_h = synthetic_pairs(BATCH, 100 + c.rank, H, W)
    a_h, b_h = a_h.pin_memory(), b_h.pin_memory()
    a_d, b_d = a_h.to(c.dev), b_h.to(c.dev)
    out_h = [torch.empty((BATCH, 2, H, W), dtype=torch.float32).pin_memory() for _ in range(2)]
    hbm, tfl, peak_kind = peaks()
    graph_pred = network.FlowPredictor(model)
    serve = network.PipelinedFlowPredictor(model, depth=2)
    ev = {}

    def hook(kind, lvl, phase):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev.setdefault((kind, lvl), []).append(e)

    def step_eager():
        return network.predict_flow(model, a_d, b_d)

    last = {}

    def step_graph():
        last["flow"] = graph_pred(a_d, b_d)

    it = [0]

    def step_e2e():
        serve.infer(a_h, b_h, out_h[it[0] & 1])
        it[0] += 1

    with torch.no_grad():
        for _ in range(max(Wm, 3)):
            step_eager()
            step_graph()
            step_e2e()
        serve.synchronize()
        # ---- value: device-resident inputs, CUDA-graph replay ----
        sampler = ClockSampler(c.local)
        sampler.start()
        torch.cuda.profiler.start()
        ms_total = timed(c, step_graph, K)
        torch.cuda.profiler.stop()
        clocks = sampler.finish()
        outputs = {k: v.cpu().numpy() for k, v in last.items()}    # the graph's output buffer: later replays overwrite it
        # ---- e2e: host buffers through the serving API; copies inside the timed region ----
        ms_e2e = timed(c, step_e2e, K, sync_extra=lambda: (torch.cuda.current_stream().wait_stream(serve.d2h),
                                                           torch.cuda.current_stream().wait_stream(serve.h2d)))
        # ---- eager pass with CUDA events around every hot-path launch (in-step kernel times) + launch count ----
        model.event_hook = hook
        n0 = _lib.launch_count()
        ms_eager = timed(c, step_eager, K)
        launches = _lib.launch_count() - n0
        model.event_hook = None
        kt = {}
        for key, lst in ev.items():
            durs = [lst[i].elapsed_time(lst[i + 1]) for i in range(0, len(lst) - 1, 2)]
            kt[key] = sum(durs) / len(durs)
        # ---- sustained: the graph loop for >= sustain seconds ----
        sust = None
        if args.sustain_seconds > 0:
            Ks = max(K, int(math.ceil(args.sustain_seconds * 1e3 / (ms_total / K))))
            s2 = ClockSampler(c.local)
            s2.start()
            ms_s = timed(c, step_graph, Ks)
            cl2 = s2.finish()
            sust = {"value": round(BATCH * Ks * c.world / (ms_s * 1e-3), 3), "unit": "pairs/s", "steps": Ks,
                    "seconds": round(ms_s * 1e-3, 3), "ms_per_step": round(ms_s / Ks, 4), "clocks": cl2}
        # ---- the dominant kernel alone, cold L2 (diagnostic) ----
        f1t = torch.randn(BATCH, 32, H // 4, W // 4, device=c.dev)
        f2t = torch.randn(BATCH, 32, H // 4, W // 4, device=c.dev)
        outb = torch.empty(BATCH, 81, H // 4, W // 4, device=c.dev)
        iso = []
        for _ in range(10):
            c.flush.zero_()
            torch.cuda._sleep(400_000)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            ops.correlation(f1t, f2t, leaky_slope=0.1, out=outb)
            g1.record()
            g1.synchronize()
            iso.append(g0.elapsed_time(g1))
        corr_kernel = _lib.last_kernel()

    pairs = BATCH * K * c.world
    value = pairs / (ms_total * 1e-3)
    # rooflines (SURVEY.md 8d): K1 bytes 4*N*H*W*(2C+81), flops 2*81*C*N*H*W; K3 bytes 4*N*H*W*3C + coarse + weights, flops 18*C^2*N*H*W
    def corr_bytes(L):
        return 4 * BATCH * (H >> L) * (W >> L) * (2 * LEVEL_C[L] + 81)

    def warp_bytes(L):
        C_ = LEVEL_C[L]
        return 4 * BATCH * (H >> L) * (W >> L) * 3 * C_ + 4 * BATCH * (H >> (L + 1)) * (W >> (L + 1)) * 3 + 4 * (9 * C_ * C_ + C_)

    def warp_flops(L):
        return 18 * LEVEL_C[L] ** 2 * BATCH * (H >> L) * (W >> L)
    t2 = kt.get(("corr", 2))
    achieved = corr_bytes(2) / (t2 * 1e-3) / 1e9 if t2 else None
    traffic, traffic_src = dram_traffic(corr_kernel)
    corr_levels = {f"L{L}": {"ms": round(kt[("corr", L)], 5), "alg_bytes": corr_bytes(L),
                             "gbs": round(corr_bytes(L) / kt[("corr", L)] / 1e6, 1),
                             "frac": round(corr_bytes(L) / kt[("corr", L)] / 1e6 / hbm, 4)} for L in (6, 5, 4, 3, 2) if ("corr", L) in kt}
    corr_sum_ms = sum(kt[("corr", L)] for L in (6, 5, 4, 3, 2) if ("corr", L) in kt)
    k3 = {f"L{L}": {"ms": round(kt[("warp", L)], 5), "alg_bytes": warp_bytes(L), "flops": warp_flops(L),
                    "gbs": round(warp_bytes(L) / kt[("warp", L)] / 1e6, 1),
                    "frac_hbm": round(warp_bytes(L) / kt[("warp", L)] / 1e6 / hbm, 4),
                    "tflops": round(warp_flops(L) / kt[("warp", L)] / 1e9, 2),
                    "frac_bf16_x3": round(3 * warp_flops(L) / kt[("warp", L)] / 1e9 / tfl, 4)} for L in (5, 4, 3, 2) if ("warp", L) in kt}
    hot_ms = sum(kt.values())
    config = {"workload": "MaskFlownet-S full 6-level forward, batch 8 per GPU, 1024x448 synthetic uint8 pairs, random-init "
                          "weights -- BASELINE configs[1]",
              "arithmetic": ARITH, "global_batch": BATCH * c.world,
              "parallelism": f"replicas x{c.world} (no data-path collective)",
              "l2": "256 MiB buffer overwritten before every step (inside the timed region, ~0.05 ms/step)",
              "value_path": "network.FlowPredictor: the step replayed from a CUDA graph, device-resident uint8 inputs",
              "e2e_path": "network.PipelinedFlowPredictor.infer: pinned host uint8 in -> H2D on a copy stream -> graph replay -> "
                          "D2H of the fp32 flow on a copy stream -> pinned host; double-buffered, all copies complete inside "
                          "the timed region",
              "eager_path": "network.predict_flow with CUDA events around every correlation / warp launch (per-kernel in-step "
                            "times, launch count); ms_per_step_eager below"}
    line = base_line(METRIC, value, K, max(Wm, 3), ms_total, c.world, config)
    line["e2e"] = {"value": round(pairs / (ms_e2e * 1e-3), 3), "unit": "pairs/s",
                   "h2d_bytes_per_step": int(a_h.numel() + b_h.numel()), "d2h_bytes_per_step": int(out_h[0].numel() * 4),
                   "ms_per_step": round(ms_e2e / K, 4)}
    line["gpu_launches"] = int(launches)      # our kernels per K eager steps; the graph replays the same launches
    line["ms_per_step_eager"] = round(ms_eager / K, 4)
    line["clocks"] = clocks
    if sust:
        line["value_sustained"] = sust
    line["roofline"] = {"kernel": f"{corr_kernel} (level-2 correlation, N=8 C=32 112x256, md=4)", "bound": "hbm",
                        "achieved": round(achieved, 1) if achieved else None, "peak": hbm, "unit": "GB/s",
                        "frac": round(achieved / hbm, 4) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                        "peak_source": peak_kind, "alg_bytes_per_launch": corr_bytes(2),
                        "launch_ms_in_step": round(t2, 5) if t2 else None,
                        "launch_ms_isolated_cold_l2": round(sum(iso) / len(iso), 5),
                        "corr_levels": corr_levels, "corr_sum_ms": round(corr_sum_ms, 5),
                        "k3_warp_levels": k3, "bf16_peak_tflops": tfl,
                        "hot_path_ms_per_step": round(hot_ms, 4), "hot_path_share_of_step": round(hot_ms / (ms_eager / K), 4)}
    if c.rank == 0 and c.world == 1 and args.cpu_sample_steps > 0:
        host_threads = usable_host_threads()
        try:
            val, sec, used = cpu_arm(args.cpu_sample_steps, 1, host_threads)
            line["cpu_baseline"] = {"value": round(val, 4), "unit": "pairs/s", "cores": used, "kind": "port",
                                    "sample": f"{args.cpu_sample_steps} steps x 1 pair at 1024x448 on {used} of "
                                              f"{host_threads} host threads (oracle/network_ref.py)"}
            line["cpu_baseline"]["corr_table"] = cpu_corr_table(host_threads)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "pairs/s", "cores": host_threads, "kind": "port",
                                    "sample": f"failed: {e}"}
    if c.rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if c.world > 1:
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------------------------------------- configs[2], [3], [4]
def bench_other(args, K, Wm):
    from maskflownet_b200 import _lib, losses, network
    c = setup_gpu()
    cfg = args.config
    torch.manual_seed(0)
    if cfg == "cascade":
        H, W, BATCH = 448, 1024, 4
        metric = "image-pairs/sec (MaskFlownet cascade forward, 1024x448)"
        workload = "MaskFlownet full cascade (S head + dual pyramid, md=2 correlations) forward, batch 4, 1024x448 -- BASELINE configs[3]"
        model = network.MaskFlownet().to(c.dev).eval()
    elif cfg == "fwdbwd":
        H, W, BATCH = 384, 512, 8
        metric = "image-pairs/sec (MaskFlownet-S forward+backward, 512x384)"
        workload = "MaskFlownet-S forward + MultiscaleEpe + backward (corr / warp grad kernels), batch 8, 512x384 -- BASELINE configs[2]"
        model = network.MaskFlownetS().to(c.dev).train()
    else:
        H, W, BATCH = 576, 960, 4
        metric = "image-pairs/sec (MaskFlownet-S training step, 960x540 padded to 960x576)"
        workload = ("MaskFlownet-S training step (fwd + bwd + one NCCL gradient all-reduce + Adam), batch 4 per GPU "
                    f"(global {4 * c.world}), 960x540 padded to 960x576 as do_batch_mx does -- BASELINE configs[4]")
        model = network.MaskFlownetS().to(c.dev).train()
    if args.train_tc_forward >= 0:
        model.train_tc_forward = bool(args.train_tc_forward)
    a_h, b_h = synthetic_pairs(BATCH, 100 + c.rank, H, W)
    a_h, b_h = a_h.pin_memory(), b_h.pin_memory()
    a_d, b_d = a_h.to(c.dev), b_h.to(c.dev)
    g = torch.Generator().manual_seed(7 + c.rank)
    flow_h = (torch.randn(BATCH, 2, H, W, generator=g) * 3).pin_memory()
    flow_d = flow_h.to(c.dev)
    mask_d = torch.ones(BATCH, 1, H, W, device=c.dev)
    loss_h = torch.empty(BATCH, dtype=torch.float32).pin_memory()
    extra = {}
    t_ar = []

    if cfg == "cascade":
        out_h = torch.empty((BATCH, 2, H, W), dtype=torch.float32).pin_memory()

        def step(x1, x2, fl):
            with torch.no_grad():
                return network.predict_flow(model, x1, x2)

        def finish(res):
            out_h.copy_(res, non_blocking=True)
        d2h = out_h.numel() * 4
    else:
        bucket = c.mdist.GradBucket(model.parameters())
        opt = torch.optim.Adam(model.parameters(), lr=1e-4) if cfg == "train8" else None     # network/pipeline.py:27

        def step(x1, x2, fl):
            bucket.zero_()
            a, b, _ = network.centralize(x1.float() / 255.0, x2.float() / 255.0)
            preds, _, _ = model(a, b)
            per_sample = losses.multiscale_epe(fl, mask_d, preds)
            per_sample.sum().backward()                  # per-sample losses are summed (pipeline.py:112-113)
            if cfg == "train8":
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                bucket.allreduce_(global_batch=BATCH * c.world)       # trainer.step(batch_size) (pipeline.py:114)
                e1.record()
                t_ar.append((e0, e1))
                opt.step()
            return per_sample.detach()

        def finish(res):
            loss_h.copy_(res, non_blocking=True)
        d2h = loss_h.numel() * 4
        extra["grad_bucket_mb"] = round(bucket.numel * 4 / 1e6, 1)

    last = {}

    def step_resident():
        last["flow" if cfg == "cascade" else "per_sample_loss"] = step(a_d, b_d, flow_d)

    def step_e2e():
        x1, x2 = a_h.to(c.dev, non_blocking=True), b_h.to(c.dev, non_blocking=True)
        fl = flow_h.to(c.dev, non_blocking=True) if cfg != "cascade" else None
        finish(step(x1, x2, fl))

    for _ in range(max(Wm, 3)):
        step_resident()
        step_e2e()
    t_ar.clear()
    sampler = ClockSampler(c.local)
    sampler.start()
    n0 = _lib.launch_count()
    torch.cuda.profiler.start()           # ncu --profile-from-start off: the launch list of the timed region only
    ms_total = timed(c, step_resident, K)
    torch.cuda.profiler.stop()
    launches = _lib.launch_count() - n0
    outputs = {k: v.cpu().numpy() for k, v in last.items()}
    if cfg != "cascade":
        outputs["grad"] = bucket.flat.cpu().numpy()       # every p.grad is a view into the bucket (parameter order)
    ar_ms = sum(x.elapsed_time(y) for x, y in t_ar) / len(t_ar) if t_ar else None
    ms_e2e = timed(c, step_e2e, K)
    clocks = sampler.finish()
    pairs = BATCH * K * c.world
    tc_fwd = bool(getattr(model, "train_tc_forward", False))
    config = {"workload": workload, "arithmetic": ARITH if cfg == "cascade" else
              "forward/backward of the hot path (correlation, fused warp): our exact-fp32 / bf16-split kernels; 3x3 convolutions: "
              + ("forward on the tcgen05 kernel (f32 I/O, bf16 hi/lo split MMA, fp32 accumulate), backward aten.convolution_backward "
                 "(cuDNN fp32, TF32 off)" if tc_fwd else "torch autograd both ways (cuDNN fp32, TF32 off)")
              + "; MultiscaleEpe: fused forward / backward kernels (csrc/loss.cu)",
              "train_tc_forward": tc_fwd,
              "global_batch": BATCH * c.world,
              "parallelism": (f"data parallel x{c.world}: batch sharded, one NCCL all-reduce of the flat fp32 gradient bucket per step"
                              if cfg == "train8" else f"replicas x{c.world}"),
              "l2": "256 MiB buffer overwritten before every step (inside the timed region)",
              "e2e_path": "pinned host uint8 pairs (+ fp32 flow labels) H2D, step, D2H of the per-sample loss (or the flow) inside the timed region"}
    line = base_line(metric, pairs / (ms_total * 1e-3), K, max(Wm, 3), ms_total, c.world, config)
    h2d = a_h.numel() + b_h.numel() + (flow_h.numel() * 4 if cfg != "cascade" else 0)
    line["e2e"] = {"value": round(pairs / (ms_e2e * 1e-3), 3), "unit": "pairs/s", "h2d_bytes_per_step": int(h2d),
                   "d2h_bytes_per_step": int(d2h), "ms_per_step": round(ms_e2e / K, 4)}
    line["gpu_launches"] = int(launches)
    line["clocks"] = clocks
    if ar_ms is not None:
        extra["grad_allreduce_ms"] = round(ar_ms, 4)
        extra["nccl_ranks"] = c.world
    line.update(extra)
    if c.rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if c.world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="fwd", choices=["fwd", "fwdbwd", "cascade", "train8"])
    ap.add_argument("--cpu-sample-steps", type=int, default=32)   # ~10 s of host work on a 16-thread box
    ap.add_argument("--sustain-seconds", type=float, default=3.0)
    ap.add_argument("--train-tc-forward", type=int, default=-1,
                    help="fwdbwd / train8: 1 = the 3x3 convolutions' forward on the tcgen05 kernel (cuDNN backward), 0 = cuDNN "
                         "both ways, -1 = the model's default")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(float32; rank 0): fwd and cascade the flow; fwdbwd and train8 the per-sample loss and the "
                         "gradient of every parameter, flattened in parameter order (train8: after the all-reduce)")
    args = ap.parse_args()
    K, Wm = args.steps, max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    host_threads = usable_host_threads()

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's outputs: it needs --impl ours")
        if rank != 0:
            return
        val, sec, used = cpu_arm(max(1, K), max(1, min(Wm, 1)), host_threads)
        line = {"impl": "reference", "metric": "image-pairs/sec (MaskFlownet-S forward, 1024x448)", "value": round(val, 4),
                "unit": "pairs/s", "n_gpus": args.gpus, "steps": K, "warmup": Wm, "ms_per_step": round(sec * 1e3, 2),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "MaskFlownet-S full 6-level forward, 1024x448 synthetic, random-init weights "
                                       "(BASELINE configs[1]); CPU sample: 1 pair per step"},
                "cpu_baseline": {"value": round(val, 4), "unit": "pairs/s", "cores": used, "kind": "port",
                                 "sample": f"{max(1, K)} steps x 1 pair at 1024x448 (oracle/network_ref.py: torch-CPU "
                                           "convs + C-oracle OpenMP correlation/deformable conv)"},
                "e2e": {"value": round(val, 4), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    if args.config == "fwd":
        bench_fwd(args, K, Wm)
    else:
        bench_other(args, K, Wm)


if __name__ == "__main__":
    main()
