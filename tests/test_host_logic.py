"""CPU: host-side logic that needs no GPU — weight packing layouts, shard arithmetic, and the
data-parallel gather over a 2-process gloo group (the same code path NCCL drives on GPUs)."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import hf_oracle
from vit import packing
from vit.parallel import DataParallelVIT, all_gather_rows, shard_bounds
from vit.utils import transfer_pretrained_weights
from vit.vit import VIT


def test_shard_bounds_cover_and_partition():
    for total in (0, 1, 7, 256, 1024, 2048, 1000):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_bounds(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            for (a, b), (c, d) in zip(spans, spans[1:]):
                assert b == c and b >= a
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(AssertionError):
        shard_bounds(4, 2, 2)


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_packed_qkv_layout_matches_hf(arch):
    """pack_attention rebuilds HF's fused (out, in) Q/K/V matrices from the per-head parameters."""
    hf = hf_oracle.build_hf(arch, seed=0)
    model = VIT(**hf_oracle.vit_kwargs(arch))
    transfer_pretrained_weights(hf, model, verbose=False)
    hsd = hf.state_dict()
    for l, block in enumerate(model.encoder.layer):
        pk = block.attention.packed()
        pre = f"encoder.layer.{l}.attention.attention."
        want_w = torch.cat([hsd[pre + f"{p}.weight"] for p in ("query", "key", "value")], dim=0)
        want_b = torch.cat([hsd[pre + f"{p}.bias"] for p in ("query", "key", "value")], dim=0)
        assert torch.equal(pk.wqkv, want_w) and torch.equal(pk.bqkv, want_b)
        assert torch.equal(pk.wo, hsd[f"encoder.layer.{l}.attention.output.dense.weight"])
        mlp = block.packed()
        assert torch.equal(mlp.w1, hsd[f"encoder.layer.{l}.intermediate.dense.weight"])
        assert torch.equal(mlp.w2, hsd[f"encoder.layer.{l}.output.dense.weight"])
    emb = model.embeddings.packed()
    K = 3 * model.patch_size ** 2
    assert emb.ldw % 8 == 0 and emb.ldw >= K
    assert torch.equal(emb.w[:, :K], hsd["embeddings.patch_embeddings.projection.weight"].reshape(-1, K))
    assert torch.count_nonzero(emb.w[:, K:]) == 0
    pos = hsd["embeddings.position_embeddings"][0]
    assert torch.allclose(emb.posb[0], pos[0] + hsd["embeddings.cls_token"].reshape(-1))
    assert torch.allclose(emb.posb[1:], pos[1:] + hsd["embeddings.patch_embeddings.projection.bias"])


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_uint8_packing_folds_the_image_processor(arch):
    """pack_embeddings_u8: raw bytes against the re-ordered, scaled weight + shifted bias table equal
    the patch projection of the rescaled / normalised pixels (what the uint8 kernel path computes)."""
    a = hf_oracle.ARCHS[arch]
    model = VIT(**hf_oracle.vit_kwargs(arch))
    with torch.no_grad():
        for p_ in model.parameters():
            p_.copy_(torch.randn_like(p_) * 0.05)
    emb = model.embeddings
    mean, std, r = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225), 1.0 / 255.0
    pk = packing.pack_embeddings_u8(emb, mean, std, r)
    S, P, D = a["image_size"], a["patch_size"], a["hidden_size"]
    g = torch.Generator().manual_seed(5)
    x = torch.randint(0, 256, (2, S, S, 3), generator=g, dtype=torch.uint8)
    # patches of the NHWC bytes in (i, j, c) order: [B, n, P*P*3]
    n = S // P
    patches = x.float().reshape(2, n, P, n, P, 3).permute(0, 1, 3, 2, 4, 5).reshape(2, n * n, P * P * 3)
    got = patches @ pk.w[:, :pk.K].float().t() + pk.posb[1:]
    xn = (x.float() * r - torch.tensor(mean)) / torch.tensor(std)
    want = torch.nn.functional.conv2d(xn.permute(0, 3, 1, 2), emb.projection.weight.float(),
                                      emb.projection.bias.float(), stride=P).flatten(2).transpose(1, 2)
    want = want + emb.position_embeddings.float()[0, 1:]
    assert torch.allclose(got, want, atol=2e-3, rtol=1e-4), (got - want).abs().max()
    assert torch.allclose(pk.posb[0], (emb.cls_token.float().reshape(-1) + emb.position_embeddings.float()[0, 0]))


def test_pooler_weights_load_transposed():
    """VIT(add_pooling_layer=True): pooler.dense is filled from HF's (out, in) weight as (in, out); the
    default model has no pooler and keeps the reference's 990-key state dict."""
    from transformers import ViTConfig, ViTModel
    arch = "tiny-b"
    torch.manual_seed(1)
    hf = ViTModel(ViTConfig(**hf_oracle.ARCHS[arch]), add_pooling_layer=True).eval()
    model = VIT(**hf_oracle.vit_kwargs(arch), add_pooling_layer=True)
    transfer_pretrained_weights(hf, model, verbose=False)
    assert torch.equal(model.pooler.dense.weight, hf.pooler.dense.weight.t())
    assert torch.equal(model.pooler.dense.bias, hf.pooler.dense.bias)
    plain = VIT(**hf_oracle.vit_kwargs(arch))
    assert plain.pooler is None and not any(k.startswith("pooler") for k in plain.state_dict())


def test_classifier_head_loads_from_image_classification_model():
    """VIT(num_labels=...): classifier.{weight,bias} are filled from HF ViTForImageClassification (source
    keys carry the ``vit.`` prefix; the (out, in) weight lands as (in, out)); the default model has no
    classifier and keeps the reference's state-dict keys."""
    from transformers import ViTConfig, ViTForImageClassification
    arch = "tiny-b"
    torch.manual_seed(2)
    hf = ViTForImageClassification(ViTConfig(**hf_oracle.ARCHS[arch], num_labels=24)).eval()
    with torch.no_grad():
        hf.classifier.weight.copy_(torch.randn_like(hf.classifier.weight))
        hf.classifier.bias.copy_(torch.randn_like(hf.classifier.bias))
    model = VIT(**hf_oracle.vit_kwargs(arch), num_labels=24)
    transfer_pretrained_weights(hf, model, verbose=False)
    assert torch.equal(model.classifier.weight, hf.classifier.weight.t())
    assert torch.equal(model.classifier.bias, hf.classifier.bias)
    assert torch.equal(model.layernorm.weight, hf.vit.layernorm.weight)
    plain = VIT(**hf_oracle.vit_kwargs(arch))
    assert plain.classifier is None and not any(k.startswith("classifier") for k in plain.state_dict())
    with pytest.raises(AssertionError):
        plain.logits(torch.zeros(1, 3, 64, 64))


def test_packed_cache_invalidation():
    model = VIT(**hf_oracle.vit_kwargs("tiny-b"))
    mha = model.encoder.layer[0].attention
    first = mha.packed()
    assert mha.packed() is first                      # cached
    with torch.no_grad():
        mha.attention[1].key.weight.add_(1.0)         # in-place update bumps the version counter
    second = mha.packed()
    assert second is not first and not torch.equal(second.wqkv, first.wqkv)
    model.load_state_dict(model.state_dict())         # load_state_dict drops the cache
    assert mha.packed() is not second
    model.to(torch.bfloat16)                          # _apply drops it and the dtype follows
    assert mha.packed().wqkv.dtype == torch.bfloat16 and mha.packed().bqkv.dtype == torch.float32


class _FakePooled(torch.nn.Module):
    """Stands in for VIT on CPU: pooled(x) = per-image mean of the pixels, (B, 3)."""

    def pooled(self, x):
        return x.mean(dim=(2, 3))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dp_worker(rank, world, port, total, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(0)
        full = torch.randn(total, 3, 4, 4, generator=g)
        dp = DataParallelVIT(_FakePooled())
        lo, hi = dp.local_slice(total)
        got = dp(full[lo:hi], total)
        torch.save(got, os.path.join(out_dir, f"rank{rank}.pt"))
        rows = all_gather_rows(torch.full((hi - lo, 2), float(rank)), total)
        torch.save(rows, os.path.join(out_dir, f"rows{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _dp_disagree_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dp = DataParallelVIT(_FakePooled())
        x = torch.randn(4, 3, 4, 4)
        # every rank claims a different global batch: the collective plan must refuse on EVERY rank
        try:
            dp(x, 8 + rank)
            verdict = "no error"
        except AssertionError as exc:
            verdict = "assert: " + str(exc)
        # ... and a consistent call afterwards still works (nothing is left half-built), also pipelined
        got = dp(x, 8)
        prev = dp.submit(x, 8)
        last = dp.flush()
        ok = prev is None and torch.equal(last, got) and got.shape == (8, 3) and dp.gather_impl == "torch.distributed"
        with open(os.path.join(out_dir, f"verdict{rank}.txt"), "w") as f:
            f.write(f"{verdict}|{ok}")
    finally:
        dist.destroy_process_group()


def test_data_parallel_plan_is_collective_gloo_world2(tmp_path):
    """The gather plan (peer-store kernel or torch.distributed, and with which shapes) is agreed through one
    all-reduce the first time a shape is seen: ranks that disagree on the global batch all raise."""
    world = 2
    mp.spawn(_dp_disagree_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        verdict, ok = open(tmp_path / f"verdict{r}.txt").read().split("|")
        assert verdict.startswith("assert: Ranks disagree on the global batch"), verdict
        assert ok == "True"


@pytest.mark.parametrize("total", [8, 7])      # equal shards (single-buffer path) and ragged shards
def test_data_parallel_gather_gloo_world2(tmp_path, total):
    world = 2
    mp.spawn(_dp_worker, args=(world, _free_port(), total, str(tmp_path)), nprocs=world, join=True)
    g = torch.Generator().manual_seed(0)
    full = torch.randn(total, 3, 4, 4, generator=g)
    want = full.mean(dim=(2, 3))
    for r in range(world):
        got = torch.load(tmp_path / f"rank{r}.pt")
        assert torch.equal(got, want), f"rank {r} gathered embeddings differ from the single-process result"
        rows = torch.load(tmp_path / f"rows{r}.pt")
        lo0, hi0 = shard_bounds(total, world, 0)
        assert torch.equal(rows[:hi0], torch.zeros(hi0, 2)) and torch.equal(rows[hi0:], torch.ones(total - hi0, 2))


def test_gelu_polynomial_restatement_matches_exact_erf():
    """The fc1 epilogue's GELU (csrc/common.cuh: gelu_erf_poly_x2) restated in fp32 numpy:
    gelu(x) = relu(x) - 0.5|x| * 2^P(|x|), P a degree-5 polynomial for log2(erfc(a/sqrt(2))).
    Must stay within 1e-6 absolute of the exact-erf GELU the reference computes
    (vit/kernels/activations.py:19-20) and underflow cleanly for large |x|."""
    import numpy as np
    coef = [np.float32(c) for c in (-0.00048810223, 0.0071987188, -0.052146632, -0.45959586, -1.1510005)]
    x = np.concatenate([np.linspace(-12, 12, 200001), [-1e4, -40.0, 0.0, 40.0, 1e4]]).astype(np.float32)
    a = np.abs(x)
    p = coef[0] * a + coef[1]
    for c in coef[2:]:
        p = p * a + c
    p = p * a
    assert (p <= 0).all()                                   # the exponential can never overflow
    with np.errstate(over="ignore", under="ignore"):
        e = np.exp2(p.astype(np.float64))
    got = np.maximum(x, 0).astype(np.float64) - 0.5 * a.astype(np.float64) * e
    want = torch.nn.functional.gelu(torch.from_numpy(x).double()).numpy()
    assert np.isfinite(got).all()
    assert np.abs(got - want).max() <= 1e-6


@pytest.mark.parametrize("K,N", [(128, 96), (768, 320), (1280, 64)])
def test_zero_sum_layernorm_fold_packing(K, N):
    """The arithmetic of the LayerNorm -> GEMM fold (csrc/ln_fold.cu restated in torch,
    oracle/fold_restatement.py; reference pair layernorm.py:90-127 + matmul.py:111-156; the GPU tests compare
    the kernel with this restatement): the folded bf16 weight rows sum to ~0, no element moves by
    more than one extra bf16 ulp, and rstd * (x @ W'^T) + b' reproduces LayerNorm -> dense as well as the
    column-sum form does."""
    import math
    torch.manual_seed(K + N)
    ln = torch.nn.LayerNorm(K, eps=1e-12)
    with torch.no_grad():
        ln.weight.copy_(1 + 0.2 * torch.randn(K))
        ln.bias.copy_(0.2 * torch.randn(K))
    w = (torch.randn(N, K) / math.sqrt(K)).bfloat16()
    b = torch.randn(N)
    from oracle import fold_restatement
    wz, bz = fold_restatement.fold_layernorm_zero_sum(w, b, ln)
    wf, bf, cs = fold_restatement.fold_layernorm_colsum(w, b, ln)
    assert wz.dtype == torch.bfloat16 and torch.equal(bz, bf)
    assert wz.double().sum(dim=1).abs().max().item() <= 2e-3 * wz.float().abs().mean().item()
    exact = w.float() * ln.weight.detach()[None, :]
    exact = exact - exact.mean(dim=1, keepdim=True)
    ulp = torch.exp2(torch.floor(torch.log2(exact.abs().clamp_min(1e-30))) - 7.0)
    assert ((wz.float() - exact).abs() <= 2.6 * ulp + 1e-12).all()     # rounding (0.5) + one move (1) + binade edges
    x = (2.0 * torch.randn(300, K) + 0.7).bfloat16().float()
    want = torch.nn.functional.layer_norm(x, (K,), ln.weight, ln.bias, 1e-12) @ w.float().t() + b
    mean = x.mean(dim=1, keepdim=True)
    rstd = (x.var(dim=1, unbiased=False, keepdim=True) + 1e-12).rsqrt()
    got_z = rstd * (x @ wz.float().t()) + bz
    got_c = rstd * (x @ wf.float().t()) - rstd * mean * cs + bf
    err_z = ((got_z - want).norm() / want.norm()).item()
    err_c = ((got_c - want).norm() / want.norm()).item()
    assert err_z <= 1.1 * err_c + 1e-5 and err_z <= 2e-3


def test_bench_dump_outputs_float32_and_bounded(tmp_path):
    """bench.py --dump-outputs: the rows exactly, in float32, while they fit in 64 MB; above that the same seeded
    sample of rows on every run, and the file stays within 64 MB."""
    import numpy as np
    import bench
    small = torch.randn(256, 768).bfloat16()
    bench.dump_pooled(str(tmp_path / "small"), small)
    got = np.load(tmp_path / "small" / "pooled.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())
    big = torch.randn(24000, 768)
    for d in ("a", "b"):
        bench.dump_pooled(str(tmp_path / d), big)
    a, b = np.load(tmp_path / "a" / "pooled.npy"), np.load(tmp_path / "b" / "pooled.npy")
    assert os.path.getsize(tmp_path / "a" / "pooled.npy") <= 64 << 20
    assert np.array_equal(a, b) and a.shape == (21844, 768)         # (64 MB - 4 KB of header) / 3 KB rows
    # every stored row is one whole row of the output, each at most once, in the output's order
    where = {r.tobytes(): i for i, r in enumerate(big.numpy())}
    idx = [where.get(r.tobytes(), -1) for r in a]
    assert min(idx) >= 0 and all(i < j for i, j in zip(idx, idx[1:]))
