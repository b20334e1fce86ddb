#!/usr/bin/env python
"""Benchmark of the hot path: ViT forward, images/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5] [--impl reference] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE for N > 1).  A step = one forward
of the per-GPU batch (c2 / c3: weak scaling, the per-GPU batch is fixed; c4 / c5: the named GLOBAL batch
divided by N) + CLS pooling + the all-gather of the pooled embeddings when N > 1 (one pool +
peer-store kernel over NVLink, vit/parallel.py:PeerGather, pipelined: step i hands its rows to the
peers and collects step i - 1, the last step is drained inside the timed region; VT_PEER_GATHER=0 =
vt_pool_cls + NCCL; `config.gather` says which ran).  The step is replayed from a CUDA graph (the
reference's own contract, vit/utils.py:115-133; `config.launch` says so, --no-graph = eager).
Rank 0 prints ONE JSON line.

  value     device-resident inputs, CUDA-event timed, max over ranks
  e2e       same steps through the public API from PINNED HOST buffers: H2D of every step's pixels
            and D2H of its pooled embeddings inside the timed region (double-buffered copy stream)
  roofline  the tcgen05 GEMM kernel (95 % of the FLOPs): algorithmic FLOPs / CUDA-event time of its
            launches, against MEASURED_PEAKS.json (burst figure for a timed region under 1 s, sustained
            above; both fractions are printed); `roofline.kernels` = the same for every kernel of the
            step (attention against the tensor AND the exp/MUFU bound, patch embedding and LayerNorm in
            GB/s).  The events are recorded in a SECOND, eager pass over the same K steps so that the
            timed region of `value` holds nothing but the steps
            `roofline.library_same_shape` (N = 1): every GEMM shape of the layer through our kernel and through
            cuBLASLt, back to back in the same process (same box, same power cap): the library comparison that
            does not depend on which peak figure the fraction is taken of
  --dump-outputs DIR    after the timed steps, DIR/pooled.npy (float32) holds what the last timed step returned:
            the pooled CLS embeddings, (global batch, hidden).  The weights and pixels are seeded, so two builds run
            with the same arguments can be compared output for output
  gather_check (N > 1)  one untimed step: peer-store gather == NCCL gather == single-process forward
  other_configs         short untimed-side measurements of the other BASELINE configs on the same box
  cpu_baseline / --impl reference
            HuggingFace ViTModel fp32 on the box's host cores (the oracle and timing reference
            BASELINE.json names; the reference's own Triton kernels cannot run on a CPU).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

CONFIGS = {
    # name: (arch, batch, "per_gpu" | "global", description).  c2 / c3 are quoted per GPU (weak scaling: the
    # metric's config is 256 images on ONE B200); c4 / c5 name a GLOBAL batch sharded over the GPUs
    # (1024 / N and 2048 / N images per GPU).
    "c2": ("vit-b16-224", 256, "per_gpu", "ViT-B/16@224 bf16 forward, batch 256 per GPU (BASELINE configs[1])"),
    "c3": ("vit-b16-384", 128, "per_gpu", "ViT-B/16@384 (577 tokens) bf16 forward, batch 128 per GPU (BASELINE configs[2])"),
    "c4": ("vit-l16-224", 1024, "global", "ViT-L/16@224 bf16 forward, global batch 1024 sharded over the GPUs (BASELINE configs[3])"),
    "c5": ("vit-h14-224", 2048, "global", "ViT-H/14@224 bf16 forward, global batch 2048 sharded over the GPUs (BASELINE configs[4])"),
}


def per_gpu_batch(config: str, world: int) -> int:
    _, batch, kind, _ = CONFIGS[config]
    if kind == "global":
        assert batch % world == 0, f"{config}: global batch {batch} does not divide over {world} GPUs"
        return batch // world
    return batch


def flops_per_image(a):
    """Algorithmic FLOPs (2*MAC) of GEMMs + attention per image (SURVEY.md 8d)."""
    D, L, F, P, S = a["hidden_size"], a["num_hidden_layers"], a["intermediate_size"], a["patch_size"], a["image_size"]
    n = (S // P) ** 2
    N = n + 1
    return 2 * n * 3 * P * P * D + L * (2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D + 4 * N * D * F)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"burst": p.get("bf16_tflops"), "sustained": p.get("bf16_tflops_sustained"),
                "hbm": p.get("hbm_gbs"), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx, power = [], set(), None, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx = float(parts[1])
                    power.append(float(parts[2]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            busy = [c for c, p in zip(sm, power) if p > 0.5 * max(power)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(power))
        return out


def hf_cpu_images_per_sec(arch, batch, budget_s=15.0):
    """HF ViTModel fp32 forward on the host cores, a bounded sample of about ``budget_s`` seconds:
    returns (img/s from the median forward, threads, list of forward times)."""
    import torch
    from oracle import hf_oracle
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, OSError):
        torch.set_num_threads(os.cpu_count() or 1)
    model = hf_oracle.build_hf(arch, seed=0)
    x = hf_oracle.make_input(arch, batch)
    times = []
    with torch.no_grad():
        t0 = time.perf_counter()
        hf_oracle.hf_forward(model, x)            # warm-up, also sizes the sample
        first = time.perf_counter() - t0
        reps = max(3, min(200, int(budget_s / max(first, 1e-3))))
        for _ in range(reps):
            t0 = time.perf_counter()
            hf_oracle.hf_forward(model, x)
            times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return batch / med, torch.get_num_threads(), times


def run_reference(args, arch, desc):
    """--impl reference: the CPU implementation of the path (HF ViTModel fp32), bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import hf_oracle
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm runs on rank 0 alone and is
    # meant to use every host thread it can
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, OSError):
        torch.set_num_threads(os.cpu_count() or 1)
    sample_batch = 32
    model = hf_oracle.build_hf(arch, seed=0)
    x = hf_oracle.make_input(arch, sample_batch)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 3))):
            hf_oracle.hf_forward(model, x)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            hf_oracle.hf_forward(model, x)
        dt = time.perf_counter() - t0
    ms = dt / args.steps * 1e3
    value = sample_batch / (ms / 1e3)
    threads = torch.get_num_threads()
    sample = f"HF ViTModel fp32 CPU forward (oracle/hf_oracle.py), {sample_batch} images per step"
    line = {
        "impl": "reference", "metric": "images_per_sec", "value": value, "unit": "img/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "arch": arch, "sample_images_per_step": sample_batch},
        "cpu_baseline": {"value": value, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def build_model(arch, dev, dtype):
    """Random-init weights of the named architecture (no network for checkpoints), same on all ranks."""
    import torch
    from vit import configs
    from vit.vit import VIT
    torch.manual_seed(0)
    model = VIT(**configs.vit_kwargs(arch))
    with torch.no_grad():
        for p in model.parameters():
            if p.dim() > 1:
                torch.nn.init.trunc_normal_(p, std=0.02)
            else:
                p.copy_(torch.randn_like(p) * 0.02)
        for m in model.modules():
            if type(m).__name__ == "LayerNormTriton":
                m.weight.add_(1.0)
    return model.to(device=dev, dtype=dtype).eval()


def classify_launch(name, args):
    """(label, flops, bytes) of one C-ABI call from its argument tuple (include/vitb200.h order)."""
    if name == "vt_gemm_bf16":
        M, N, K, gelu, res = args[10], args[11], args[12], args[13], args[8]
        return f"gemm N={N} K={K}" + ("+gelu" if gelu else "") + ("+res" if res else ""), 2.0 * M * N * K, None
    if name == "vt_gemm_bf16_ln":
        M, N, K, gelu, res, rs, so = args[9], args[10], args[11], args[12], args[7], args[13], args[17]
        tag = ("+ln" if rs else "") + ("+gelu" if gelu else "") + ("+res" if res else "") + ("+stats" if so else "")
        return f"gemm N={N} K={K}{tag}", 2.0 * M * N * K, None
    if name == "vt_flash_attn":
        B, H, N, dh = args[4], args[5], args[6], args[7]
        return f"attention N={N} dh={dh}", 4.0 * B * H * N * N * dh, None
    if name in ("vt_patch_embed", "vt_patch_embed_stats"):
        o = 1 if name == "vt_patch_embed_stats" else 0
        pix_dtype, B, C, S, P, D = args[1], args[7 + o], args[8 + o], args[9 + o], args[10 + o], args[11 + o]
        es = {0: 4, 1: 2, 2: 1}[pix_dtype]
        n = (S // P) ** 2
        return "patch_embed", 2.0 * B * n * C * P * P * D, float(B) * (C * S * S * es + (n + 1) * D * 2) + C * P * P * D * 2
    if name == "vt_patch_embed_gemm":      # gather + token-mode GEMM, timed as one unit
        pix_dtype, B, C, S, P, D = args[1], args[9], args[10], args[11], args[12], args[13]
        es = {0: 4, 1: 2, 2: 1}[pix_dtype]
        n = (S // P) ** 2
        return "patch_embed", 2.0 * B * n * C * P * P * D, float(B) * (C * S * S * es + (n + 1) * D * 2) + C * P * P * D * 2
    if name == "vt_gemm_fp8":
        M, N, K = args[11], args[12], args[13]
        return f"gemm_fp8 N={N} K={K}", 2.0 * M * N * K, None
    if name == "vt_layernorm_fp8":
        return "layernorm_fp8", None, float(args[4]) * args[5] * 3
    if name == "vt_layernorm":
        rows, dim, in_dt, out_dt = args[4], args[5], args[9], args[10]
        return "layernorm", None, float(rows) * dim * ({0: 4, 1: 2}[in_dt] + {0: 4, 1: 2}[out_dt])
    if name == "vt_pool_cls":
        return "pool_cls", None, 2.0 * args[2] * args[3] * 2
    if name == "vt_pool_cls_allgather":
        return "pool_cls_allgather", None, None
    return name, None, None


class KernelTimer:
    """CUDA events around every launch issued through vit.kernels._lib.call (eager passes only)."""

    def __init__(self):
        self.records = []      # (label, flops, bytes, ev0, ev1)
        self._open = None

    def hook(self, name, before, args):
        import torch
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        if before:
            self._open = (classify_launch(name, args), ev)
        else:
            (label, flops, nbytes), ev0 = self._open
            self.records.append((label, flops, nbytes, ev0, ev))

    def summary(self):
        agg = {}
        for label, flops, nbytes, ev0, ev1 in self.records:
            a = agg.setdefault(label, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            a["launches"] += 1
            a["ms"] += ev0.elapsed_time(ev1)
            a["flops"] += flops or 0.0
            a["bytes"] += nbytes or 0.0
        return agg


def roofline_kernels(agg, peaks, tensor_peak, sm_mhz, steps):
    """Per-kernel roofline entries from a KernelTimer summary."""
    out = []
    for label, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        sec = a["ms"] / 1e3
        e = {"kernel": label, "launches_per_step": a["launches"] / steps, "avg_launch_us": a["ms"] * 1e3 / a["launches"],
             "ms_per_step": a["ms"] / steps}
        if label.startswith("gemm_fp8"):
            tf = a["flops"] / sec / 1e12
            e.update(bound="tensor", achieved=tf, peak=2 * tensor_peak, unit="TFLOP/s", frac=tf / (2 * tensor_peak),
                     peak_note="fp8 dense = 2 x the measured bf16 figure (nominal ratio; no measured fp8 peak on file)")
        elif label.startswith("gemm"):
            tf = a["flops"] / sec / 1e12
            e.update(bound="tensor", achieved=tf, peak=tensor_peak, unit="TFLOP/s", frac=tf / tensor_peak)
        elif label.startswith("attention"):
            tf = a["flops"] / sec / 1e12
            # one exponential per score: flops / (4 dh); the MUFU pipe issues 16 per clock and SM
            dh = int(label.split("dh=")[1])
            exps = a["flops"] / (4.0 * dh) / sec
            mufu_peak = 16.0 * 148 * (sm_mhz or 1965.0) * 1e6
            e.update(bound="tensor", achieved=tf, peak=tensor_peak, unit="TFLOP/s", frac=tf / tensor_peak,
                     exp_per_s=exps, exp_peak_per_s=mufu_peak, frac_of_exp_bound=exps / mufu_peak,
                     exp_peak_note="16 ex2 per clock per SM x 148 SMs at the SM clock sampled during the run")
        elif label == "patch_embed":
            # gather (HBM) + token-mode GEMM (tensor), timed as one unit: the binding bound is whichever of
            # bytes / HBM peak and FLOPs / tensor peak is the longer (the GEMM: 59 GFLOP against 165 MB at C2)
            gbs = a["bytes"] / sec / 1e9
            tf = a["flops"] / sec / 1e12
            if tf / tensor_peak >= gbs / peaks["hbm"]:
                e.update(bound="tensor", achieved=tf, peak=tensor_peak, unit="TFLOP/s", frac=tf / tensor_peak,
                         hbm_gbs=gbs, frac_of_hbm_peak=gbs / peaks["hbm"])
            else:
                e.update(bound="hbm", achieved=gbs, peak=peaks["hbm"], unit="GB/s", frac=gbs / peaks["hbm"], tflops=tf)
        elif a["bytes"]:
            gbs = a["bytes"] / sec / 1e9
            e.update(bound="hbm", achieved=gbs, peak=peaks["hbm"], unit="GB/s", frac=gbs / peaks["hbm"])
        out.append(e)
    return out


class StepRunner:
    """One step of the data-parallel forward, replayed from a CUDA graph per input buffer when possible."""

    def __init__(self, dp, world, global_batch, use_graph):
        self.dp, self.world, self.global_batch = dp, world, global_batch
        self.use_graph = use_graph
        self.graphs = {}
        self.launches_per_graph = 0
        self.note = "eager launches"

    def eager(self, x):
        if self.world > 1:
            return self.dp.submit(x, self.global_batch)
        return self.dp(x)

    def finish(self):
        """Collect the last step's gathered rows (pipelined gather); None on one GPU."""
        return self.dp.flush() if self.world > 1 else None

    def capture(self, buffers):
        import torch
        from vit.kernels import _lib
        if not self.use_graph:
            return
        if self.world > 1 and self.dp.gather_impl != "peer-store kernel":
            self.note = "eager launches (NCCL gather is not captured)"
            return
        try:
            if self.world > 1 and not self.dp._pending:
                self.eager(buffers[0])     # the captured step must contain the collect of its predecessor
                torch.cuda.synchronize()
            pool = torch.cuda.graph_pool_handle()   # the graphs run one after the other: one activation pool
            for b in buffers:
                n0 = _lib.launch_count
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    out = self.eager(b)
                self.launches_per_graph = _lib.launch_count - n0
                self.graphs[b.data_ptr()] = (g, out)
            self.note = f"CUDA-graph replay ({self.launches_per_graph} kernel launches per graph)"
        except Exception as exc:   # capture refused: fall back to eager launches and say so
            self.graphs = {}
            self.note = f"eager launches (graph capture failed: {type(exc).__name__})"
            torch.cuda.synchronize()

    def __call__(self, x):
        hit = self.graphs.get(x.data_ptr())
        if hit is None:
            return self.eager(x)
        hit[0].replay()
        return hit[1]

    def launches(self, steps, eager_count):
        return self.launches_per_graph * steps if self.graphs else eager_count


def quick_config(name, world, rank, dev, steps=5, warmup=3, fp8=False):
    """Short device-resident measurement of another BASELINE config on the same box (side field);
    ``fp8``: with the optional FP8 path (e4m3 QKV / fc1 / fc2 GEMMs) switched on for the measurement."""
    import torch
    from vit import configs
    from vit import vit as vit_mod
    from vit.parallel import DataParallelVIT
    arch = CONFIGS[name][0]
    batch = per_gpu_batch(name, world)
    a = configs.ARCHS[arch]
    model = build_model(arch, dev, torch.bfloat16)
    dp = DataParallelVIT(model)
    S = a["image_size"]
    g = torch.Generator().manual_seed(99 + rank)
    xs = [torch.randn((batch, 3, S, S), generator=g).to(torch.bfloat16).to(dev) for _ in range(2)]
    run = StepRunner(dp, world, batch * world, use_graph=False)
    vit_mod.set_fp8(fp8)
    try:
        with torch.no_grad():
            for i in range(warmup):
                run(xs[i & 1])
            run.finish()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                run(xs[i & 1])
            run.finish()
            e1.record()
            torch.cuda.synchronize()
    finally:
        vit_mod.set_fp8(False)
    ms = e0.elapsed_time(e1) / steps
    del model, dp, xs
    torch.cuda.empty_cache()
    return {"arch": arch, "per_gpu_batch": batch, "global_batch": batch * world, "ms_per_step": ms, "steps": steps,
            "flops_per_image": flops_per_image(a)}


def c1_fp32_latency(dev, reps=20):
    """BASELINE configs[0] on the GPU: ViT-B/16@224 fp32, batch 1 — a latency figure (ms per image)."""
    import torch
    model = build_model("vit-b16-224", dev, torch.float32)
    x = torch.randn(1, 3, 224, 224, device=dev)
    with torch.no_grad():
        for _ in range(3):
            model(x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            model(x)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del model
    torch.cuda.empty_cache()
    return {"arch": "vit-b16-224", "dtype": "f32", "batch": 1, "ms_per_image": ms, "img_s": 1e3 / ms, "reps": reps}


def library_same_shape(dev, M, D, F, secs=0.3):
    """Untimed side measurement for the roofline object: the four GEMM shapes of a layer, each run back to back for
    ``secs`` seconds through OUR kernel (with its fused epilogue) and through cuBLASLt (torch.addmm: bias only)
    in the same process, i.e. the same box and the same power cap.  The measured peak in MEASURED_PEAKS.json is
    cuBLAS on 8192^3; this says what the library reaches on the shapes the model actually runs."""
    import math
    import torch
    from vit.kernels import _lib
    out_rows = []
    for (K, N, gelu, res, what) in ((D, 3 * D, 0, False, "qkv"), (D, F, 1, False, "fc1 + GELU"),
                                    (D, D, 0, True, "out-proj + residual"), (F, D, 0, True, "fc2 + residual")):
        x = torch.randn(M, K, device=dev).bfloat16()
        w = (torch.randn(N, K, device=dev) / math.sqrt(K)).bfloat16()
        bias = torch.randn(N, device=dev)
        bias16 = bias.bfloat16()
        r = torch.randn(M, N, device=dev).bfloat16() if res else None
        out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)

        def ours():
            _lib.call("vt_gemm_bf16", x.data_ptr(), K, w.data_ptr(), K, out.data_ptr(), N, _lib.VT_BF16, bias.data_ptr(),
                      None if r is None else r.data_ptr(), N, M, N, K, gelu, _lib.stream_ptr(x))

        def lib():
            torch.addmm(bias16, x, w.t(), out=out)

        res_tf = []
        for fn in (ours, lib):
            for _ in range(10):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                fn()
            e1.record()
            torch.cuda.synchronize()
            n = max(20, int(secs * 1e3 / (e0.elapsed_time(e1) / 20)))
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res_tf.append(2.0 * M * N * K * n / (e0.elapsed_time(e1) / 1e3) / 1e12)
        out_rows.append({"shape": f"M={M} N={N} K={K}", "ours_tflops": res_tf[0], "ours_epilogue": what,
                         "cublaslt_tflops": res_tf[1], "cublaslt_epilogue": "bias", "ours_over_library": res_tf[0] / res_tf[1]})
        del x, w, r, out
    return {"note": f"each shape back to back for {secs} s per implementation, same process (same box, same power cap); "
                    "cuBLASLt through torch.addmm", "shapes": out_rows}


def dump_pooled(out_dir, rows):
    """``out_dir``/pooled.npy: the rows in float32, or the same seeded sample of them on every run when all of
    them would take more than 64 MB."""
    import numpy as np
    import torch
    cap = ((64 << 20) - 4096) // (4 * rows.shape[1])      # 4 KB left for the .npy header
    if rows.shape[0] > cap:
        pick = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:cap]
        rows = rows[pick.sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pooled.npy"), rows.float().numpy())


def gather_check(model, dp, x, global_batch, world, rank):
    """One untimed step three ways: peer-store kernel, NCCL all-gather, and (rank 0) the single-process
    forward of the first images of every rank's shard.  Returns a dict of verdicts (identical on all ranks)."""
    import torch
    import torch.distributed as dist
    from vit.parallel import DataParallelVIT
    with torch.no_grad():
        a = dp(x, global_batch).clone()
        via_nccl = DataParallelVIT(model, peer_gather=False)(x, global_batch)
        k = min(8, x.shape[0])
        heads = torch.empty((world * k,) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
        dist.all_gather_into_tensor(heads, x[:k].contiguous())
        whole = model.pooled(heads)
        rows = torch.cat([a[r * x.shape[0]: r * x.shape[0] + k] for r in range(world)], dim=0)
    ok = torch.tensor([int(torch.equal(a, via_nccl)), int(torch.equal(rows, whole))], device=x.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    ok = ok.tolist()
    return {"gather": dp.gather_impl, "vs_nccl_all_gather": "bit-equal" if ok[0] else "MISMATCH",
            "vs_single_process_forward": ("bit-equal" if ok[1] else "MISMATCH") +
            f" (first {k} images of every rank's shard recomputed in one process on each rank)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the side measurements of the other BASELINE configs")
    ap.add_argument("--profile-step", action="store_true",
                    help="bracket ONE extra eager step after the timed region with cudaProfilerStart/Stop "
                         "(ncu --profile-from-start off then captures exactly one forward)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step to DIR/pooled.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the output of the B200 path; --impl reference has none to write")
    args.warmup = max(args.warmup, 3)

    arch, _, _, desc = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, arch, desc)
        return

    import torch
    import torch.distributed as dist
    from vit import configs
    from vit.kernels import _lib
    from vit.parallel import DataParallelVIT

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    batch = args.batch or per_gpu_batch(args.config, world)
    a = configs.ARCHS[arch]
    model = build_model(arch, dev, torch.bfloat16)
    dp = DataParallelVIT(model)
    global_batch = batch * world

    # synthetic pixels: several distinct input batches are rotated so no step re-reads a cached input
    S = a["image_size"]
    n_rot = 4
    g = torch.Generator().manual_seed(1234 + rank)
    host_inputs = [torch.randn((batch, 3, S, S), generator=g).to(torch.bfloat16).pin_memory() for _ in range(n_rot)]
    dev_inputs = [h.to(dev, non_blocking=True) for h in host_inputs]
    torch.cuda.synchronize()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    run = StepRunner(dp, world, global_batch, use_graph=not args.no_graph)

    # ----------------------------------------------------------------- device-resident timing
    with torch.no_grad():
        check = gather_check(model, dp, dev_inputs[0], global_batch, world, rank) if world > 1 else None
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()          # nvidia-smi needs ~0.5 s to produce its first sample
        for i in range(args.warmup):
            run.eager(dev_inputs[i % n_rot])
        sync_all()
        run.capture(dev_inputs)
        for i in range(args.warmup):   # warm-up in the form that is timed (graph replays)
            run(dev_inputs[i % n_rot])
        run.finish()
        sync_all()
        # timed region: EXACTLY K steps (+ the drain of the last step's gather), nothing else between the events
        launches0 = _lib.launch_count
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for i in range(args.steps):
            out = run(dev_inputs[i % n_rot])
        last = run.finish()
        stop.record()
        sync_all()
        launches = run.launches(args.steps, _lib.launch_count - launches0)
        # copied now: the passes below may reuse the buffers of the timed step
        timed_rows = (last if last is not None else out).cpu() if args.dump_outputs else None
        # the same K steps again, eagerly, with a CUDA event before and after EVERY kernel launch (rooflines);
        # kept out of the region above because ~130 event records per step cost 2-4 %
        timer = KernelTimer()
        _lib.event_hook = timer.hook
        h_start, h_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h_start.record()
        for i in range(args.steps):
            out = run.eager(dev_inputs[i % n_rot])
        run.finish()
        h_stop.record()
        _lib.event_hook = None
        sync_all()
        clocks = sampler.stop() if rank == 0 else None
    if args.profile_step:
        with torch.no_grad():
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            run.eager(dev_inputs[0])
            run.finish()
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
    ms_total = start.elapsed_time(stop)
    hooked_ms_total = h_start.elapsed_time(h_stop)
    kagg = timer.summary()
    gemm_ms = sum(v["ms"] for k, v in kagg.items() if k.startswith("gemm N"))        # the bf16 dense layers
    n_gemm = sum(v["launches"] for k, v in kagg.items() if k.startswith("gemm N"))
    kernels_ms = sum(v["ms"] for v in kagg.values())

    # ----------------------------------------------------------------- end-to-end from pinned host memory
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    pooled_host = torch.empty((global_batch, a["hidden_size"]), dtype=torch.bfloat16).pin_memory()

    def e2e_run(nsteps, hosts, devs, runner):
        cur = torch.cuda.current_stream()
        with torch.cuda.stream(copy_stream):
            devs[0].copy_(hosts[0], non_blocking=True)
            ready[0].record(copy_stream)
        for i in range(nsteps):
            slot = i & 1
            if i + 1 < nsteps:
                nxt = (i + 1) & 1
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(consumed[nxt])
                    devs[nxt].copy_(hosts[(i + 1) % n_rot], non_blocking=True)
                    ready[nxt].record(copy_stream)
            cur.wait_event(ready[slot])
            res = runner(devs[slot])
            consumed[slot].record(cur)
            if res is not None:          # pipelined gather: the rows of the previous step (None at step 0)
                pooled_host.copy_(res, non_blocking=True)
        res = runner.finish()
        if res is not None:
            pooled_host.copy_(res, non_blocking=True)

    def e2e_time(hosts, devs):
        runner = StepRunner(dp, world, global_batch, use_graph=not args.no_graph)
        with torch.no_grad():
            e2e_run(3, hosts, devs, runner)
            sync_all()
            runner.capture(devs)
            e2e_run(3, hosts, devs, runner)
            sync_all()
            e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_host0 = time.perf_counter()
            e_start.record()
            e2e_run(args.steps, hosts, devs, runner)
            e_stop.record()
            sync_all()
            wall = (time.perf_counter() - t_host0) * 1e3
        return max(e_start.elapsed_time(e_stop), 0.0), wall

    bufs = [torch.empty_like(dev_inputs[0]) for _ in range(2)]
    e2e_ms, e2e_wall_ms = e2e_time(host_inputs, bufs)
    # same steps from RAW uint8 NHWC host pixels: the image processor's rescale + normalise run inside
    # the patch-embedding kernel (VIT.forward_uint8), so the H2D copy is one byte per pixel value
    g8 = torch.Generator().manual_seed(4321 + rank)
    host_u8 = [torch.randint(0, 256, (batch, S, S, 3), generator=g8, dtype=torch.uint8).pin_memory()
               for _ in range(n_rot)]
    bufs_u8 = [torch.empty((batch, S, S, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    e2e_u8_ms, _ = e2e_time(host_u8, bufs_u8)

    # ----------------------------------------------------------------- other BASELINE configs, same box (side fields)
    others = {}
    if not args.no_other_configs and args.config == "c2" and not args.batch:
        del bufs, bufs_u8
        torch.cuda.empty_cache()
        names = ["c3"] if world == 1 else ["c4"] + (["c5"] if world == 8 else [])
        with torch.no_grad():
            for name in names:
                others[name] = quick_config(name, world, rank, dev)
            if world == 1:
                others["c1"] = c1_fp32_latency(dev)
                others["c2_fp8"] = quick_config("c2", world, rank, dev, steps=10, fp8=True)
                others["c2_fp8"]["dtype"] = "e4m3 QKV / fc1 / fc2 operands (VT_FP8=1), NOT the headline bf16 metric"

    # ----------------------------------------------------------------- reduce over ranks
    other_ms = [others[k]["ms_per_step"] for k in sorted(others) if "ms_per_step" in others[k]]
    stats = torch.tensor([ms_total, e2e_ms, gemm_ms, float(launches), e2e_u8_ms] + other_ms, device=dev, dtype=torch.float64)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_total, e2e_ms, e2e_u8_ms = mx[0].item(), mx[1].item(), mx[4].item()
        launches = int(sm[3].item())
        for k, v in zip([k for k in sorted(others) if "ms_per_step" in others[k]], mx[5:].tolist()):
            others[k]["ms_per_step"] = v
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_pooled(args.dump_outputs, timed_rows)

    ms_per_step = ms_total / args.steps
    value = global_batch * args.steps / (ms_total / 1e3)
    e2e_value = global_batch * args.steps / (e2e_ms / 1e3)
    fpi = flops_per_image(a)
    peaks = measured_peaks()
    # burst peak for a timed region shorter than about a second (the power cap has not bitten yet: the
    # driver's own burst figure is a best-of-10 of ~1 ms GEMMs), the sustained one above
    region_s = ms_total / 1e3
    use_burst = region_s < 1.0
    tensor_peak = peaks["burst"] if use_burst else peaks["sustained"]

    # GEMM FLOPs per step on this rank (QKV, proj, fc1, fc2 of every layer; patch-embed and attention
    # are separate kernels and not counted here)
    D, L, F = a["hidden_size"], a["num_hidden_layers"], a["intermediate_size"]
    N_tok = (S // a["patch_size"]) ** 2 + 1
    gemm_flops_step = L * batch * N_tok * (2 * D * 3 * D + 2 * D * D + 4 * D * F)
    gemm_tflops = gemm_flops_step * args.steps / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_dram_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    whole_tf = fpi * batch / (ms_per_step / 1e3) / 1e12
    roofline = {
        "kernel": "gemm2_bf16_kernel (tcgen05 cta_group::2)", "bound": "tensor", "achieved": gemm_tflops,
        "peak": tensor_peak, "unit": "TFLOP/s",
        "frac": (gemm_tflops / tensor_peak) if gemm_tflops else None,
        "frac_of_burst_peak": (gemm_tflops / peaks["burst"]) if gemm_tflops else None,
        "frac_of_sustained_peak": (gemm_tflops / peaks["sustained"]) if gemm_tflops else None,
        "peak_source": peaks["source"] + (f", burst figure (timed region {region_s:.2f} s < 1 s)" if use_burst else
                                          f", sustained figure (timed region {region_s:.2f} s under the power cap)"),
        "traffic": traffic, "launches_timed": n_gemm,
        "avg_launch_us": (gemm_ms / n_gemm * 1e3) if n_gemm else None,
        "algorithmic_flops_per_launch": gemm_flops_step / (4 * L),
        "share_of_step": gemm_ms / hooked_ms_total,
        "timed_in": "a second, eager pass over the same K steps with a CUDA event around every kernel launch "
                    f"({hooked_ms_total / args.steps:.3f} ms per step with the events)",
        "whole_forward_tflops": whole_tf,
        "whole_forward_frac_of_burst_peak": whole_tf / peaks["burst"],
        "whole_forward_frac_of_sustained_peak": whole_tf / peaks["sustained"],
        "kernel_time_ms_per_step": kernels_ms / args.steps,
        "launch_gap_ms_per_step": ms_per_step - kernels_ms / args.steps,
        "kernels": roofline_kernels(kagg, peaks, tensor_peak, (clocks or {}).get("sm_mhz"), args.steps),
    }
    for k, o in others.items():
        if "ms_per_step" in o:
            o["img_s"] = o["global_batch"] * 1e3 / o["ms_per_step"]
            o["whole_forward_tflops_per_gpu"] = o.pop("flops_per_image") * o["per_gpu_batch"] / (o["ms_per_step"] / 1e3) / 1e12
            o["frac_of_burst_peak"] = o["whole_forward_tflops_per_gpu"] / peaks["burst"]
            o["note"] = f"{o['steps']} eager steps after 3 warm-ups, device-resident, max over ranks"

    line = {
        "metric": "images_per_sec", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak" if CONFIGS[args.config][2] == "per_gpu" or args.batch else "strong",
        "vs_baseline": None,
        "dtype": "bf16" if os.environ.get("VT_FP8", "0") != "1" else "e4m3 QKV/fc1/fc2 operands + bf16 (VT_FP8=1: not the BASELINE metric)",
        "data": "synthetic",
        "config": {"workload": desc, "arch": arch, "per_gpu_batch": batch, "global_batch": global_batch,
                   "tokens": N_tok, "parallelism": f"dp{world}" if world > 1 else "single",
                   "l2": f"{n_rot} distinct input batches rotated; per-step activation footprint > L2",
                   "weights": "random-init (trunc-normal 0.02), replicated",
                   "launch": run.note,
                   "gather": ("pooled CLS embeddings, " + dp.gather_impl + ", pipelined (step i collects step i-1; "
                              "the last step is drained inside the timed region)") if world > 1 else "none (one GPU)"},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": "img/s", "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": host_inputs[0].numel() * 2 * world,
                "d2h_bytes_per_step": pooled_host.numel() * 2 * world,
                "host_wall_ms_per_step": e2e_wall_ms / args.steps,
                "api": "DataParallelVIT(model) steps from pinned host bf16 pixels, double-buffered H2D, D2H of the "
                       "gathered embeddings every step",
                "uint8_nhwc": {"value": global_batch * args.steps / (e2e_u8_ms / 1e3), "unit": "img/s",
                               "ms_per_step": e2e_u8_ms / args.steps,
                               "h2d_bytes_per_step": host_u8[0].numel() * world,
                               "api": "same, from pinned host RAW uint8 NHWC pixels (VIT.forward_uint8: "
                                      "rescale + normalise folded into the patch-embedding kernel)"}},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if check is not None:
        line["gather_check"] = check
    if others:
        line["other_configs"] = others
    if world == 1 and not args.no_cpu_baseline:
        cpu_val, threads, times = hf_cpu_images_per_sec(arch, 32)
        line["cpu_baseline"] = {"value": cpu_val, "unit": "img/s", "cores": threads, "kind": "port",
                                "host_cpus": os.cpu_count(),
                                "sample": f"HF ViTModel fp32 CPU forward of {arch}, batch 32, median of {len(times)} "
                                          f"forwards after 1 warm-up ({sum(times):.1f} s of CPU work)"}
    if world == 1 and not args.no_other_configs:
        try:
            line["roofline"]["library_same_shape"] = library_same_shape(dev, batch * N_tok, D, F)
        except Exception as exc:   # side measurement only
            line["roofline"]["library_same_shape"] = {"error": str(exc)[:200]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
