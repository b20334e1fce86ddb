"""Throughput of the CLIP image encoders B/32, B/16 and L/14 at 224^2 next to ViT-B/16, batch 256, bf16, each forward
replayed from a CUDA graph, one process; and the per-launch time of the fc1 GEMM at the ViT-B/16 batch-256 shape
(M = 256 * 197, N = 3072, K = 768) with the exact-GELU epilogue against the quick-GELU one.

CLIP-B/16 has ViT-B/16's shape: the same GEMMs and attention, quick GELU in fc1, one LayerNorm before block 0 in place of
the final one (``vt_layernorm_stats``, so block 0 stays folded).  The models take random-init weights drawn like
``bench.build_model``'s.  Before timing, each graph's output is checked equal to an eager forward bit for bit.  The
models alternate round by round, so slow drifts of the clock hit all of them; every round replays ``--reps`` forwards
between CUDA events.  The two fc1 epilogues alternate the same way over ``--gemm-reps`` launches per round on the same
operands.  Prints one JSON line with the device name and power limit, read in the same process; ``--out FILE`` also
writes it there.  Needs a CUDA device."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def build_clip(arch, dev, dtype):
    """Random-init CLIP image encoder of ``configs.CLIP_ARCHS``, parameters drawn as ``bench.build_model`` draws them."""
    import torch
    from vit import configs
    from vit.vit import VIT
    torch.manual_seed(0)
    model = VIT(**configs.clip_kwargs(arch))
    with torch.no_grad():
        for p in model.parameters():
            if p.dim() > 1:
                torch.nn.init.trunc_normal_(p, std=0.02)
            else:
                p.copy_(torch.randn_like(p) * 0.02)
        for m in model.modules():
            if type(m).__name__ == "LayerNormTriton":
                m.weight.add_(1.0)
        model.embeddings.projection.bias.zero_()          # CLIP's patch convolution has no bias
    return model.to(device=dev, dtype=dtype).eval()


def fc1_times(dev, rounds, reps):
    """Median microseconds per fc1 launch (vt_gemm_bf16, bias + activation epilogue) for GELU and quick GELU."""
    import torch
    from vit.kernels import _lib
    M, N, K = 256 * 197, 3072, 768
    g = torch.Generator().manual_seed(3)
    a = torch.randn((M, K), generator=g).to(dev, torch.bfloat16)
    w = (torch.randn((N, K), generator=g) * K ** -0.5).to(dev, torch.bfloat16)
    bias = torch.randn((N,), generator=g).to(dev)
    out = torch.empty((M, N), device=dev, dtype=torch.bfloat16)
    stream = _lib.stream_ptr(a)

    def launch(act):
        _lib.call("vt_gemm_bf16", a.data_ptr(), K, w.data_ptr(), K, out.data_ptr(), N, _lib.VT_BF16, bias.data_ptr(),
                  None, 0, M, N, K, act, stream)

    acts = {"gelu": _lib.VT_ACT_GELU, "quick_gelu": _lib.VT_ACT_QUICK_GELU}
    for act in acts.values():
        for _ in range(10):
            launch(act)
    torch.cuda.synchronize()
    us = {name: [] for name in acts}
    for r in range(rounds):
        for name in (list(acts) if r % 2 == 0 else list(acts)[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                launch(acts[name])
            e1.record()
            e1.synchronize()
            us[name].append(e0.elapsed_time(e1) * 1e3 / reps)
    return {name: dict(us_median=round(statistics.median(v), 2), us_min=round(min(v), 2), us_max=round(max(v), 2))
            for name, v in us.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--gemm-reps", type=int, default=50)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from bench import build_model
    from resolution_bench import device_info
    from vit.utils import capture_cuda_graph
    assert torch.cuda.is_available(), "clip_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)
    models = {"vit_b16": build_model("vit-b16-224", dev, torch.bfloat16),
              "clip_b32": build_clip("clip-b32-224", dev, torch.bfloat16),
              "clip_b16": build_clip("clip-b16-224", dev, torch.bfloat16),
              "clip_l14": build_clip("clip-l14-224", dev, torch.bfloat16)}
    g = torch.Generator().manual_seed(0)
    x = torch.randn((args.batch, 3, 224, 224), generator=g).to(dev, torch.bfloat16)

    graphs = {}
    with torch.no_grad():
        for name, model in models.items():
            static = x.clone()
            graph, out = capture_cuda_graph(model, static)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(out, model(x)), f"{name}: graph replay differs from the eager forward"
            # the graph reads `static` and writes `out` at their addresses on every replay: both live as long as it
            graphs[name] = (graph, static, out)
        rates = {name: [] for name in graphs}
        for r in range(args.rounds):
            names = list(graphs) if r % 2 == 0 else list(graphs)[::-1]
            for name in names:
                graph = graphs[name][0]
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    graph.replay()
                e1.record()
                e1.synchronize()
                rates[name].append(args.batch * args.reps / (e0.elapsed_time(e1) / 1e3))
        fc1 = fc1_times(dev, args.rounds, args.gemm_reps)

    result = dict(info, batch=args.batch, dtype="bf16", rounds=args.rounds, reps=args.reps)
    for name, values in rates.items():
        result[name] = dict(tokens=graphs[name][2].shape[1], img_per_s_median=round(statistics.median(values), 1),
                            img_per_s_min=round(min(values), 1), img_per_s_max=round(max(values), 1))
    result["clip_b16_over_vit_b16"] = round(result["clip_b16"]["img_per_s_median"] /
                                            result["vit_b16"]["img_per_s_median"], 4)
    result["fc1_c2"] = fc1
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
