"""Cost of ``output_attentions`` / ``output_hidden_states``, ViT-B/16@224 bf16 (the C2 workload: 256 images), one process.

  kernel   ``vt_attn_probs`` against ``vt_flash_attn`` on the same C2 QKV activation (B = 256, H = 12, N = 197), the two
           launches alternating round by round, ``--reps`` launches between CUDA events per round.  The probabilities'
           bytes written over the kernel's time is reported as a share of the B200's 7.7 TB/s (data sheet).  The QKV
           activation (232 MB) and the probabilities (238 MB) exceed the 126 MB L2.
  forward  the forward with the flags off, with ``output_hidden_states`` and with ``output_attentions``, as CUDA-graph
           replays alternating round by round.

Prints one JSON line with the device name and power limit read in the same call; ``--out FILE`` also writes it there.
Needs a CUDA device."""
import argparse
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

HBM_BYTES_PER_S = 7.7e12


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from mim_bench import capture
    from resolution_bench import device_info
    from vit import configs
    from vit.kernels import _lib
    from vit.vit import VIT
    assert torch.cuda.is_available(), "outputs_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)

    # ---- kernel: vt_attn_probs against vt_flash_attn on the C2 QKV
    B, N, H, dh = args.batch, 197, 12, 64
    D = H * dh
    g = torch.Generator().manual_seed(1)
    qkv = torch.randn((B, N, 3 * D), generator=g).to(dev, torch.bfloat16)
    ctx = torch.empty((B, N, D), device=dev, dtype=torch.bfloat16)
    probs = torch.empty((B, H, N, N), device=dev, dtype=torch.bfloat16)
    base, es, stream = qkv.data_ptr(), 2, _lib.stream_ptr(qkv)
    scale = 1.0 / math.sqrt(dh)
    launches = {
        "vt_flash_attn": lambda: _lib.call("vt_flash_attn", base, base + D * es, base + 2 * D * es, ctx.data_ptr(), B, H,
                                           N, dh, qkv.stride(1), qkv.stride(0), D, N * D, scale, stream),
        "vt_attn_probs": lambda: _lib.call("vt_attn_probs", base, base + D * es, probs.data_ptr(), B, H, N, dh,
                                           qkv.stride(1), qkv.stride(0), scale, stream),
    }
    for fn in launches.values():
        fn()
    torch.cuda.synchronize()
    us = {name: [] for name in launches}
    for r in range(args.rounds):
        for name in (list(launches) if r % 2 == 0 else list(launches)[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                launches[name]()
            e1.record()
            torch.cuda.synchronize()
            us[name].append(e0.elapsed_time(e1) * 1e3 / args.reps)
    probs_us = statistics.median(us["vt_attn_probs"])
    flash_us = statistics.median(us["vt_flash_attn"])
    probs_bytes = probs.numel() * 2

    # ---- forward: flags off / hidden states / attentions, CUDA-graph replays
    torch.manual_seed(0)
    model = VIT(**configs.vit_kwargs("vit-b16-224"))
    with torch.no_grad():
        for p in model.parameters():
            if p.dim() > 1:
                torch.nn.init.trunc_normal_(p, std=0.02)
            else:
                p.copy_(torch.randn_like(p) * 0.02)
        for m in model.modules():
            if type(m).__name__ == "LayerNormTriton":
                m.weight.add_(1.0)
    model = model.to(device=dev, dtype=torch.bfloat16).eval()
    x = torch.randn((B, 3, 224, 224), generator=g).to(dev, torch.bfloat16)
    with torch.no_grad():
        graphs = {
            "flags_off": capture(lambda: model(x))[0],
            "hidden_states": capture(lambda: model(x, output_hidden_states=True))[0],
            "attentions": capture(lambda: model(x, output_attentions=True))[0],
        }
        for gr in graphs.values():
            gr.replay()
        torch.cuda.synchronize()
        ms = {name: [] for name in graphs}
        for r in range(args.rounds):
            for name in (list(graphs) if r % 2 == 0 else list(graphs)[::-1]):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    graphs[name].replay()
                e1.record()
                torch.cuda.synchronize()
                ms[name].append(e0.elapsed_time(e1) / args.reps)

    def summary(r, unit):
        med = statistics.median(r)
        return {f"{unit}_median": round(med, 3), f"{unit}_min": round(min(r), 3), f"{unit}_max": round(max(r), 3),
                "spread_pct": round(100.0 * (max(r) - min(r)) / med, 2)}

    res = dict(info)
    res.update({
        "note": (f"ViT-B/16@224 bf16, batch {B}; {args.rounds} alternating rounds of {args.reps} launches / replays; "
                 "spread = (max - min) / median over rounds"),
        "kernel": {name: summary(r, "us") for name, r in us.items()},
        "attn_probs_over_flash": round(probs_us / flash_us, 3),
        "attn_probs_bytes_written": probs_bytes,
        "attn_probs_share_of_7.7TBps": round(probs_bytes / (probs_us * 1e-6) / HBM_BYTES_PER_S, 3),
        "forward": {name: summary(r, "ms") for name, r in ms.items()},
        "hidden_states_over_off": round(statistics.median(ms["hidden_states"]) / statistics.median(ms["flags_off"]), 4),
        "attentions_over_off": round(statistics.median(ms["attentions"]) / statistics.median(ms["flags_off"]), 4),
    })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
