"""Throughput of masked inputs and of the masked image modeling step, ViT-B/16@224 bf16 (the C2 workload: 256 images),
CUDA-graph replays, one process.  Three captured cases:

  unmasked   ``model(x)``: token-mode patch embedding (gather + 2-CTA GEMM with padded token rows);
  masked     ``model(x, bool_masked_pos=m)``, a random 60 % mask (SimMIM's ratio): masked gather + plain-mode GEMM
             with a per-row position table;
  mim        ``model.masked_image_modeling(x, m)``: the masked forward, the decoder GEMM over every row, and the
             pixel-shuffle reconstruction with the masked L1 loss.

The three alternate round by round (order reversed every other round), so slow drifts of the clock hit all of them;
every round times ``--reps`` replays between CUDA events.  Before timing, an all-false mask is checked to give the
unmasked output bit for bit.  Prints one JSON line with the device name and power limit read in the same call;
``--out FILE`` also writes it there.  Needs a CUDA device."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def build_mim_model(dev, dtype):
    """bench.py's random-init ViT-B/16@224 recipe, with the mask token and the SimMIM decoder."""
    import torch
    from vit import configs
    from vit.vit import VIT
    torch.manual_seed(0)
    model = VIT(**configs.vit_kwargs("vit-b16-224"), add_decoder=True)
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


def capture(fn):
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--ratio", type=float, default=0.6)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from resolution_bench import device_info
    assert torch.cuda.is_available(), "mim_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)
    model = build_mim_model(dev, torch.bfloat16)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((args.batch, 3, 224, 224), generator=g).to(dev, torch.bfloat16)
    n = model.embeddings.num_patches
    mask = (torch.rand((args.batch, n), generator=g) < args.ratio).to(dev)

    with torch.no_grad():
        none = torch.zeros_like(mask)
        assert torch.equal(model(x, bool_masked_pos=none), model(x)), "all-false mask differs from the unmasked call"
        graphs = {
            "unmasked": capture(lambda: model(x))[0],
            "masked": capture(lambda: model(x, bool_masked_pos=mask))[0],
            "mim": capture(lambda: model.masked_image_modeling(x, mask))[0],
        }
        for gr in graphs.values():
            gr.replay()
        torch.cuda.synchronize()
        rates = {name: [] for name in graphs}
        for r in range(args.rounds):
            names = list(graphs) if r % 2 == 0 else list(graphs)[::-1]
            for name in names:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    graphs[name].replay()
                e1.record()
                torch.cuda.synchronize()
                rates[name].append(args.batch * args.reps / (e0.elapsed_time(e1) / 1e3))

    def summary(r):
        med = statistics.median(r)
        return {"img_per_s_median": round(med, 1), "img_per_s_min": round(min(r), 1), "img_per_s_max": round(max(r), 1),
                "spread_pct": round(100.0 * (max(r) - min(r)) / med, 2)}

    res = dict(info)
    res.update({
        "note": (f"ViT-B/16@224 bf16, batch {args.batch}, CUDA-graph replays, {args.rounds} alternating rounds of "
                 f"{args.reps} replays, {int(args.ratio * 100)} % random mask; spread = (max - min) / median over rounds"),
        "cases": {name: summary(r) for name, r in rates.items()},
        "masked_over_unmasked": round(statistics.median(rates["masked"]) / statistics.median(rates["unmasked"]), 4),
        "mim_over_unmasked": round(statistics.median(rates["mim"]) / statistics.median(rates["unmasked"]), 4),
        "all_false_mask_bit_equal": True,
    })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
