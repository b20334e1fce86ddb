"""Cost of running a checkpoint at another input resolution (``interpolate_pos_encoding=True``), ViT-B/16 bf16, every
forward replayed from a CUDA graph, batch 128 (the C3 batch), one process:

  (a) the native vit-b16-384 model at 384 x 384 against the vit-b16-224 checkpoint at 384 x 384 with interpolation:
      both have 577 tokens and the same launches, so they should differ by no more than the run-to-run spread;
  (b) the 224 checkpoint at 384 x 384 against 288 x 512 (also 577 tokens): the rectangular patch gather;
  (c) the 224 checkpoint at 512 x 512 (1025 tokens) and 160 x 160 (101 tokens);
  (d) the one-time cost of a new resolution: position-table resample plus the derived bf16 table, in ms.

The cases of (a) and (b) alternate round by round, so slow drifts of the clock hit both; every round times
``--replays`` graph replays between CUDA events.  Prints one JSON line with the device name and power limit;
``--out FILE`` also writes it there.  Needs a CUDA device."""
import argparse
import functools
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def device_info(index: int) -> dict:
    import torch
    info = {"device": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        limit, clock = [v.strip() for v in q.stdout.strip().split(",")[:2]]
        info.update(power_limit_w=float(limit), max_sm_clock_mhz=float(clock))
    except Exception as exc:                       # the numbers are still printed, without the cap
        info["power_limit_w"] = f"unavailable ({exc!r})"
    return info


class Case:
    """One captured forward: ``model(x, interpolate_pos_encoding=interp)`` on a fixed (batch, 3, H, W) input."""

    def __init__(self, name, model, batch, hw, interp, seed):
        import torch
        from vit.utils import capture_cuda_graph
        g = torch.Generator().manual_seed(seed)
        self.name, self.hw, self.batch = name, hw, batch
        self.x = torch.randn((batch, 3) + hw, generator=g).to("cuda", torch.bfloat16)
        fn = functools.partial(model, interpolate_pos_encoding=True) if interp else model
        self.graph, self.out = capture_cuda_graph(fn, self.x)
        self.tokens = self.out.shape[1]
        self.rates = []

    def time(self, replays: int) -> float:
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(replays):
            self.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        rate = self.batch * replays / (e0.elapsed_time(e1) / 1e3)
        self.rates.append(rate)
        return rate

    def summary(self) -> dict:
        r = self.rates
        return {"hw": list(self.hw), "tokens": self.tokens, "img_per_s_median": round(statistics.median(r), 1),
                "img_per_s_min": round(min(r), 1), "img_per_s_max": round(max(r), 1),
                "spread_pct": round(100.0 * (max(r) - min(r)) / statistics.median(r), 2)}


def compare(a: Case, b: Case) -> dict:
    """Difference of the medians against the spread of either side."""
    ma, mb = statistics.median(a.rates), statistics.median(b.rates)
    diff = 100.0 * (mb - ma) / ma
    spread = max(a.summary()["spread_pct"], b.summary()["spread_pct"])
    return {"a": a.name, "b": b.name, "diff_pct": round(diff, 2), "spread_pct": round(spread, 2),
            "within_spread": abs(diff) <= spread}


def new_grid_cost_ms(model, grids) -> list:
    """Host-clocked, device-synchronised cost of the tables of a grid the model has not seen."""
    import torch
    from vit import packing
    emb = model.embeddings
    emb.packed()
    out = []
    for gh, gw in grids:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        packing.pos_grid(emb, gh, gw).table(emb, None, False)
        torch.cuda.synchronize()
        out.append(round((time.perf_counter() - t0) * 1e3, 3))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from bench import build_model
    assert torch.cuda.is_available(), "resolution_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)

    m224 = build_model("vit-b16-224", dev, torch.bfloat16)
    m384 = build_model("vit-b16-384", dev, torch.bfloat16)
    B = args.batch
    with torch.no_grad():
        native = Case("vit-b16-384 native 384x384", m384, B, (384, 384), False, 1)
        i384 = Case("vit-b16-224 interpolated 384x384", m224, B, (384, 384), True, 2)
        i288x512 = Case("vit-b16-224 interpolated 288x512", m224, B, (288, 512), True, 3)
        i512 = Case("vit-b16-224 interpolated 512x512", m224, B, (512, 512), True, 4)
        i160 = Case("vit-b16-224 interpolated 160x160", m224, B, (160, 160), True, 5)
        cases = [native, i384, i288x512, i512, i160]
        for c in cases:                                  # warm-up in the timed form
            c.time(args.replays)
            c.rates.clear()
        for r in range(args.rounds):
            order = cases if r % 2 == 0 else cases[::-1]
            for c in order:
                c.time(args.replays)
        grids = [(20, 30), (21, 17), (33, 33), (9, 40), (26, 26)]
        cost = new_grid_cost_ms(m224, grids)

    res = dict(info)
    res.update({
        "note": (f"ViT-B/16 bf16, batch {B}, CUDA-graph replays, {args.rounds} alternating rounds of {args.replays} "
                 "replays per case; spread = (max - min) / median over the rounds; one fixed input per case "
                 "(the forward's activations, not the input, dominate the traffic)"),
        "cases": {c.name: c.summary() for c in cases},
        "a_native384_vs_interpolated384": compare(native, i384),
        "b_interpolated384_vs_288x512": compare(i384, i288x512),
        "c_img_per_s": {"512x512": i512.summary()["img_per_s_median"], "160x160": i160.summary()["img_per_s_median"]},
        "d_new_resolution_ms": {"grids": [list(g) for g in grids], "ms": cost,
                                "median_ms": round(statistics.median(cost), 3)},
    })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
