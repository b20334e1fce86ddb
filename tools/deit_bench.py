"""Throughput of DeiT-B/16 against ViT-B/16 at 224^2, batch 256, bf16, each forward replayed from a CUDA graph, one
process.  DeiT-B/16 is the same encoder with a distillation token after CLS: 198 tokens per image instead of 197, the
same 224-row padding of the patch-embedding GEMM and the same attention tiles, 0.5 % more rows in every dense layer.

Both models take random-init weights (bench.build_model; the DeiT one with ``distillation_token=True`` and its token
drawn like the CLS token).  Before timing, each graph's output is checked equal to an eager forward bit for bit.  The
two alternate round by round, so slow drifts of the clock hit both; every round replays ``--reps`` forwards between CUDA
events.  Prints one JSON line with the device name and power limit, read in the same process; ``--out FILE`` also
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


def build_deit(dev, dtype):
    """ViT-B/16@224 weights of ``bench.build_model`` with a distillation token: the same parameters, the position table
    grown by one row and the token drawn like the CLS token."""
    import torch
    from bench import build_model
    from vit import configs
    from vit.vit import VIT
    vit = build_model("vit-b16-224", torch.device("cpu"), torch.float32)
    model = VIT(**configs.vit_kwargs("vit-b16-224"), distillation_token=True)
    sd = vit.state_dict()
    g = torch.Generator().manual_seed(1)
    pos = sd["embeddings.position_embeddings"]
    sd["embeddings.position_embeddings"] = torch.cat([pos[:, :1], torch.randn(pos[:, :1].shape, generator=g) * 0.02,
                                                      pos[:, 1:]], dim=1)
    sd["embeddings.distillation_token"] = torch.randn((1, 1, pos.shape[2]), generator=g) * 0.02
    model.load_state_dict(sd)
    return model.to(device=dev, dtype=dtype).eval()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch
    from bench import build_model
    from resolution_bench import device_info
    from vit.utils import capture_cuda_graph
    assert torch.cuda.is_available(), "deit_bench.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info(0)
    models = {"vit_b16": build_model("vit-b16-224", dev, torch.bfloat16), "deit_b16": build_deit(dev, torch.bfloat16)}
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

    result = dict(info, batch=args.batch, dtype="bf16", rounds=args.rounds, reps=args.reps)
    for name, values in rates.items():
        result[name] = dict(tokens=graphs[name][2].shape[1], img_per_s_median=round(statistics.median(values), 1),
                            img_per_s_min=round(min(values), 1), img_per_s_max=round(max(values), 1))
    result["deit_over_vit"] = round(result["deit_b16"]["img_per_s_median"] / result["vit_b16"]["img_per_s_median"], 4)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
