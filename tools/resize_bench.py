"""Speed of the image processor's resize on the device (``resize_uint8``: vt_resize_u8 / vt_resize_u8_list).

  kernel  256 images each of 375x500, 1080x1920 and 256x256 (x 3 channels) -> 224x224, BILINEAR, in the batch form
          (one tensor) and the list form (256 tensors: descriptors and tables uploaded on every call); ``--reps`` warm
          calls between CUDA events per case, the cases alternating over ``--rounds`` rounds.  Bytes = pixels read once +
          output written once; the share is of 7.7 TB/s (HGX B200 data sheet, one GPU).  The 256x256 batch (50 MB) fits
          in the 126 MB L2, the others do not.
  host    wall time of building the coefficient tables and uploading the descriptors of a list of 256 distinct sizes,
          with the host table cache cleared (cold) and filled (warm), up to the return of the call (no synchronise).
  c2      the C2 forward (ViT-B/16@224 bf16, batch 256) replayed from CUDA graphs: ``forward_uint8`` of a 224x224 batch,
          and ``forward_uint8(do_resize=True)`` of a 375x500 batch; the two alternate round by round.

Prints one JSON line with the device name and power limit read in the same call; ``--out FILE`` also writes it there.
Needs a CUDA device."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "vit.triton_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

HBM_BYTES_PER_S = 7.7e12


def _events_ms(fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--graph-reps", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from mim_bench import build_mim_model, capture
    from resolution_bench import device_info
    from vit.kernels import resize as rz
    from vit.kernels import resize_uint8
    assert torch.cuda.is_available(), "resize_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = dict(device_info(0))
    B, S = args.batch, 224
    g = torch.Generator(device=dev).manual_seed(0)

    # ---- kernel
    batches = {f"{h}x{w}": torch.randint(0, 256, (B, h, w, 3), generator=g, dtype=torch.uint8, device=dev)
               for h, w in [(375, 500), (1080, 1920), (256, 256)]}
    cases = {}
    for name, x in batches.items():
        lst = list(x.unbind(0))
        assert torch.equal(resize_uint8(x, S, S), resize_uint8(lst, S, S)), name
        cases[f"batch {name}"] = (lambda x=x: resize_uint8(x, S, S), x.numel())
        cases[f"list {name}"] = (lambda lst=lst: resize_uint8(lst, S, S), x.numel())
    for fn, _ in cases.values():
        for _ in range(3):
            fn()
    times = {name: [] for name in cases}
    for r in range(args.rounds):
        for name in (list(cases) if r % 2 == 0 else list(cases)[::-1]):
            times[name].append(_events_ms(cases[name][0], args.reps))
    out_bytes = B * S * S * 3
    kernel = {}
    for name, (_, in_bytes) in cases.items():
        ms = statistics.median(times[name])
        moved = in_bytes + out_bytes
        kernel[name] = {"us_per_call": round(ms * 1e3, 2), "spread_pct": round(100 * (max(times[name]) - min(times[name])) / ms, 2),
                        "bytes_moved": moved, "tb_per_s": round(moved / (ms / 1e3) / 1e12, 3),
                        "share_of_7.7TBps": round(moved / (ms / 1e3) / HBM_BYTES_PER_S, 3)}
    res["kernel"] = kernel
    del batches, cases
    torch.cuda.empty_cache()

    # ---- host: tables and descriptors of 256 distinct sizes
    sizes = [(300 + i, 400 + 2 * i) for i in range(B)]
    imgs = [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8, device=dev) for h, w in sizes]
    torch.cuda.synchronize()
    host = {}
    for label in ("cold", "warm", "warm2"):
        if label == "cold":
            rz._table_cached.cache_clear()
        t0 = time.perf_counter()
        resize_uint8(imgs, S, S)
        host[label + "_ms"] = round((time.perf_counter() - t0) * 1e3, 3)
        torch.cuda.synchronize()
    res["host_256_distinct_sizes"] = host
    del imgs

    # ---- the C2 forward from CUDA graphs, with and without the resize in front
    model = build_mim_model(dev, torch.bfloat16)
    x224 = torch.randint(0, 256, (B, S, S, 3), generator=g, dtype=torch.uint8, device=dev)
    x375 = torch.randint(0, 256, (B, 375, 500, 3), generator=g, dtype=torch.uint8, device=dev)
    with torch.no_grad():
        assert torch.equal(model.forward_uint8(x375, do_resize=True), model.forward_uint8(resize_uint8(x375, S, S)))
        graphs = {"forward_uint8 224x224": capture(lambda: model.forward_uint8(x224))[0],
                  "forward_uint8 375x500 do_resize": capture(lambda: model.forward_uint8(x375, do_resize=True))[0]}
        ms = {name: [] for name in graphs}
        for r in range(args.rounds):
            for name in (list(graphs) if r % 2 == 0 else list(graphs)[::-1]):
                ms[name].append(_events_ms(graphs[name].replay, args.graph_reps))
    res["c2_graph"] = {name: {"ms_per_forward": round(statistics.median(v), 3),
                              "img_per_s": round(B / (statistics.median(v) / 1e3), 1),
                              "spread_pct": round(100 * (max(v) - min(v)) / statistics.median(v), 2)}
                       for name, v in ms.items()}
    res["note"] = (f"batch {B} -> {S}x{S}, BILINEAR; kernel: median over {args.rounds} alternating rounds of {args.reps} "
                   f"calls; c2: {args.graph_reps} graph replays per round")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
