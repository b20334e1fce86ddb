"""Throughput of a batch of images at different resolutions, ViT-B/16@224 bf16, eager (a ragged call cannot be
captured into a CUDA graph, so no case uses one), one process.  One fixed list of ``--images`` images spread over the
grids of ``SIZES`` in a seeded random order, run three ways:

  ragged     ``model.forward_ragged(list)``: one packed activation, one launch per dense layer, one attention launch
             per distinct token count;
  per grid   one ``model(x, interpolate_pos_encoding=True)`` call per resolution on the stacked images of that size
             (the stacking is not timed);
  per image  one ``model(x[None], interpolate_pos_encoding=True)`` call per image.

The three alternate round by round, so slow drifts of the clock hit all of them; every round times ``--reps`` passes
over the list between CUDA events.  Before timing, the ragged outputs are checked equal to the per-image ones bit for
bit.  Prints one JSON line with the device name and power limit; ``--out FILE`` also writes it there.  Needs a CUDA
device."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# the trained grid and six others: more than the four grids packing.pos_grid keeps for single-resolution calls
SIZES = [(224, 224), (240, 320), (384, 256), (256, 256), (160, 192), (320, 240), (288, 288)]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from bench import build_model
    from resolution_bench import device_info
    assert torch.cuda.is_available(), "ragged_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)
    model = build_model("vit-b16-224", dev, torch.bfloat16)

    g = torch.Generator().manual_seed(0)
    which = torch.randint(0, len(SIZES), (args.images,), generator=g).tolist()
    images = [torch.randn((3,) + SIZES[k], generator=g).to(dev, torch.bfloat16) for k in which]
    stacks = [torch.stack([im for im, k in zip(images, which) if k == s]) for s in range(len(SIZES)) if s in which]
    tokens = sum(1 + (h // 16) * (w // 16) for h, w in (SIZES[k] for k in which))

    def ragged():
        model.forward_ragged(images)

    def per_grid():
        for x in stacks:
            model(x, interpolate_pos_encoding=True)

    def per_image():
        for x in images:
            model(x[None], interpolate_pos_encoding=True)

    cases = {"ragged": ragged, "per_grid": per_grid, "per_image": per_image}
    rates = {name: [] for name in cases}
    with torch.no_grad():
        got = model.forward_ragged(images)
        for i in range(0, len(images), max(1, len(images) // 16)):
            want = model(images[i][None], interpolate_pos_encoding=True)[0]
            assert torch.equal(got[i], want), f"image {i}: ragged output differs from its own call"
        for fn in cases.values():                        # warm-up of every shape in the timed form
            fn()
        torch.cuda.synchronize()
        for r in range(args.rounds):
            names = list(cases) if r % 2 == 0 else list(cases)[::-1]
            for name in names:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    cases[name]()
                e1.record()
                torch.cuda.synchronize()
                rates[name].append(args.images * args.reps / (e0.elapsed_time(e1) / 1e3))

    def summary(r):
        med = statistics.median(r)
        return {"img_per_s_median": round(med, 1), "img_per_s_min": round(min(r), 1), "img_per_s_max": round(max(r), 1),
                "spread_pct": round(100.0 * (max(r) - min(r)) / med, 2)}

    res = dict(info)
    res.update({
        "note": (f"ViT-B/16@224 bf16, eager, {args.images} images over {len(stacks)} resolutions ({tokens} tokens), "
                 f"{args.rounds} alternating rounds of {args.reps} passes; spread = (max - min) / median over rounds"),
        "sizes": [list(SIZES[s]) for s in range(len(SIZES)) if s in which],
        "images_per_size": [len(x) for x in stacks],
        "cases": {name: summary(r) for name, r in rates.items()},
        "ragged_over_per_grid": round(statistics.median(rates["ragged"]) / statistics.median(rates["per_grid"]), 3),
        "ragged_over_per_image": round(statistics.median(rates["ragged"]) / statistics.median(rates["per_image"]), 3),
    })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
