"""GPU parity of the whole forward against HuggingFace ViTModel (the oracle BASELINE.json names).

Tolerances (BASELINE.json north_star / SURVEY.md 8c): fp32 <= 1e-3 max-abs on the final hidden
states; bf16 cosine >= 0.999 and max-abs <= 0.15 (HF's own bf16 CPU forward differs from its fp32 by
7.1e-2 / 0.99993)."""
import os

import pytest
import torch

from oracle import hf_oracle, restatement

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _build(arch, dtype, hf=None):
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    hf = hf or hf_oracle.build_hf(arch, seed=0)
    model = VIT(**hf_oracle.vit_kwargs(arch))
    transfer_pretrained_weights(hf, model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval(), hf


def _cos(a, b):
    return torch.nn.functional.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_tiny_fp32_matches_golden(arch, golden_dir):
    gold = torch.load(os.path.join(golden_dir, f"hf_{arch}.pt"))
    hf = hf_oracle.build_hf_golden(gold)
    model, _ = _build(arch, torch.float32, hf)
    with torch.no_grad():
        got = model(hf_oracle.golden_input(gold).to(DEV)).cpu()
    assert (got - gold["output"]).abs().max().item() <= 1e-4


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_tiny_bf16_matches_golden(arch, golden_dir):
    gold = torch.load(os.path.join(golden_dir, f"hf_{arch}.pt"))
    hf = hf_oracle.build_hf_golden(gold)
    model, _ = _build(arch, torch.bfloat16, hf)
    with torch.no_grad():
        got = model(hf_oracle.golden_input(gold).to(DEV, torch.bfloat16)).float().cpu()
    assert _cos(got, gold["output"]) >= 0.999
    assert (got - gold["output"]).abs().max().item() <= 0.15


def test_c1_vit_b16_fp32_batch1_matches_hf(golden_dir):
    """BASELINE config 0: ViT-B/16@224 batch 1 fp32 vs HF ViTModel on CPU, <= 1e-3 max-abs."""
    model, hf = _build("vit-b16-224", torch.float32)
    x = hf_oracle.make_input("vit-b16-224", 2)
    want = hf_oracle.hf_forward(hf, x)
    gold = torch.load(os.path.join(golden_dir, "hf_vit-b16-224.pt"))
    if str(torch.__version__) == gold["torch"]:
        assert (want[:, gold["tokens"]] - gold["output"]).abs().max().item() <= 1e-5
    with torch.no_grad():
        got1 = model(x[:1].to(DEV)).cpu()
        got2 = model(x.to(DEV)).cpu()
    assert (got1 - want[:1]).abs().max().item() <= 1e-3
    assert (got2 - want).abs().max().item() <= 1e-3
    # the oracle restatement agrees too (same custom state-dict)
    sd = {k: v.cpu() for k, v in model.state_dict().items()}
    assert (restatement.vit_forward(sd, x[:1]) - got1).abs().max().item() <= 1e-3


def test_c2_vit_b16_bf16_matches_hf():
    """BASELINE config 1 arithmetic (bf16) on a slice of the batch the CPU oracle finishes quickly."""
    model, hf = _build("vit-b16-224", torch.bfloat16)
    x = hf_oracle.make_input("vit-b16-224", 4)
    want = hf_oracle.hf_forward(hf, x)
    with torch.no_grad():
        got = model(x.to(DEV, torch.bfloat16)).float().cpu()
    assert torch.isfinite(got).all()
    assert _cos(got, want) >= 0.999, f"cosine {_cos(got, want)}"
    assert (got - want).abs().max().item() <= 0.15, f"max-abs {(got - want).abs().max().item()}"
    for i in range(4):
        assert _cos(got[i], want[i]) >= 0.999


def test_batch_independence_full_batch_c2():
    """Full C2 batch (256): every image's output equals the output it gets in a batch of 4 —
    a size-independent property standing in for the oracle at sizes it cannot reach quickly.  All 64
    slices: at 256 images every GEMM group and attention CTA walks many tiles, so a wrong later tile
    shows up here as one slice that differs."""
    model, _ = _build("vit-b16-224", torch.bfloat16)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(256, 3, 224, 224, generator=g).to(DEV, torch.bfloat16)
    with torch.no_grad():
        full = model(x)
        for lo in range(0, 256, 4):
            part = model(x[lo:lo + 4].contiguous())
            assert torch.equal(full[lo:lo + 4], part), f"images {lo}..{lo+3} differ between batch 256 and batch 4"


def test_c3_vit_b16_384_bf16_matches_hf():
    model, hf = _build("vit-b16-384", torch.bfloat16)
    x = hf_oracle.make_input("vit-b16-384", 2)
    want = hf_oracle.hf_forward(hf, x)
    with torch.no_grad():
        got = model(x.to(DEV, torch.bfloat16)).float().cpu()
    assert _cos(got, want) >= 0.999 and (got - want).abs().max().item() <= 0.15


def test_unfused_path_matches_fused():
    """set_fused(False) runs the reference-structured per-head path through the individual entry
    points; both paths must agree (fp32: tightly)."""
    from vit import vit as vit_mod
    model, hf = _build("tiny-b", torch.float32)
    x = hf_oracle.make_input("tiny-b", 2).to(DEV)
    with torch.no_grad():
        fused = model(x)
        vit_mod.set_fused(False)
        try:
            unfused = model(x)
        finally:
            vit_mod.set_fused(True)
    assert (fused - unfused).abs().max().item() <= 1e-4


def test_cuda_graph_replay_equals_eager():
    from vit.utils import capture_cuda_graph
    model, _ = _build("tiny-b", torch.bfloat16)
    x = hf_oracle.make_input("tiny-b", 4).to(DEV, torch.bfloat16)
    with torch.no_grad():
        eager = model(x).clone()
    static_in = x.clone()
    graph, static_out = capture_cuda_graph(model, static_in)
    static_in.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, eager)


def test_launch_modes_are_bit_identical(tmp_path):
    """The GEMM launched as preferred clusters of four with the shared operand TMA-multicast + programmatic dependent
    launch (the default) computes bit for bit what plain clusters of two launched one after the other compute
    (VT_GEMM_QUAD=0 VT_PDL=0), eagerly and replayed from a CUDA graph; the bounded-logit attention path differs from the
    exact one by rounding only.  The switches are read once per process: three worker processes."""
    import subprocess
    import sys
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "launch_mode_worker.py")
    results = {}
    for tag, env in (("default", {}), ("plain", {"VT_GEMM_QUAD": "0", "VT_PDL": "0"}), ("exact", {"VT_ATTN_NO_BOUND": "1"})):
        path = str(tmp_path / f"{tag}.pt")
        e = dict(os.environ)
        for k in ("VT_GEMM_QUAD", "VT_PDL", "VT_ATTN_NO_BOUND"):
            e.pop(k, None)
        e.update(env)
        proc = subprocess.run([sys.executable, worker, path], env=e, capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stderr[-2000:]
        results[tag] = torch.load(path)
    d, pl, ex = results["default"], results["plain"], results["exact"]
    assert set(d) == set(pl) and len(d) >= 6
    for k in d:
        assert torch.isfinite(d[k].float()).all(), k
        assert torch.equal(d[k], pl[k]), f"{k}: clusters of four / dependent launch differ from the plain launch"
    assert torch.equal(d["eager"], d["graph"])
    err = (d["eager"].float() - ex["eager"].float()).abs().max().item()
    assert 0.0 <= err <= 5e-2, f"bounded-logit attention vs exact softmax: max-abs {err}"


def test_repack_after_weight_update():
    model, _ = _build("tiny-b", torch.bfloat16)
    x = hf_oracle.make_input("tiny-b", 2).to(DEV, torch.bfloat16)
    with torch.no_grad():
        before = model(x).clone()
        sd = {k: v * 1.5 if k.endswith("query.weight") else v for k, v in model.state_dict().items()}
        model.load_state_dict(sd)
        after = model(x)
    assert not torch.equal(before, after)


def test_layernorm_folding_matches_unfolded_and_hf():
    """Folding LayerNorm into the GEMM epilogues changes the launch sequence, not the result: both
    variants stay within the bf16 tolerance of HF and agree closely with each other."""
    from vit import vit as vit_mod
    model, hf = _build("vit-b16-224", torch.bfloat16)
    x = hf_oracle.make_input("vit-b16-224", 3)
    want = hf_oracle.hf_forward(hf, x)
    xd = x.to(DEV, torch.bfloat16)
    results = {}
    try:
        with torch.no_grad():
            for name, (fold, mlp) in {"plain": (False, False), "qkv": (True, False), "both": (True, True)}.items():
                vit_mod.set_layernorm_folding(fold, mlp=mlp)
                results[name] = model(xd).float().cpu()
                assert torch.equal(results[name], model(xd).float().cpu())   # statistics are exchanged without atomics
    finally:
        vit_mod.set_layernorm_folding(True, mlp=True)     # the defaults
    plain = results["plain"]
    for name, got in results.items():
        assert _cos(got, want) >= 0.999 and (got - want).abs().max().item() <= 0.15, name
    for name in ("qkv", "both"):
        folded = results[name]
        assert _cos(folded, plain) >= 0.9995, name
        assert (folded - want).abs().max().item() <= 1.5 * (plain - want).abs().max().item() + 0.02, name


@pytest.mark.parametrize("arch", ["vit-l16-224", "vit-h14-224"])
def test_c4_c5_architectures_bf16_match_hf(arch):
    """BASELINE configs 3 / 4 (ViT-L/16, ViT-H/14: 14-pixel patches, K = 588, dh = 80, 257 tokens) at
    full width and depth on the two images the CPU oracle finishes in seconds."""
    model, hf = _build(arch, torch.bfloat16)
    x = hf_oracle.make_input(arch, 2)
    want = hf_oracle.hf_forward(hf, x)
    with torch.no_grad():
        got = model(x.to(DEV, torch.bfloat16)).float().cpu()
    assert torch.isfinite(got).all()
    assert _cos(got, want) >= 0.999, f"cosine {_cos(got, want)}"
    assert (got - want).abs().max().item() <= 0.15, f"max-abs {(got - want).abs().max().item()}"


def _plant_outliers(hf, kind):
    """Make a random-init HF model produce the activations real checkpoints have (and N(0, 1) inputs through
    random weights do not): massive-activation channels in the residual stream and rows whose mean is
    large against their spread."""
    with torch.no_grad():
        layers = hf.encoder.layer
        D = layers[0].output.dense.bias.numel()
        if kind in ("massive_channels", "both"):
            # a few residual-stream channels pushed to +-40..150 by the MLP output bias of the first blocks
            for i, (ch, v) in enumerate(((5, 60.0), (D // 2 + 3, -120.0), (D - 7, 150.0), (130 % D, -40.0))):
                layers[min(i, len(layers) - 1) // 2].output.dense.bias[ch] += v
        if kind in ("large_mean", "both"):
            # every channel of every token shifted: |mean| / std of the rows entering block 0 is ~ 6 .. 8
            hf.embeddings.position_embeddings += 4.0
            layers[0].attention.output.dense.bias += 2.0
    return hf


@pytest.mark.parametrize("kind", ["massive_channels", "large_mean", "both"])
@pytest.mark.parametrize("arch", ["tiny-b", "vit-b16-224"])
def test_layernorm_folding_with_planted_outliers(arch, kind):
    """The default-on LayerNorm fold (one launch chain: statistics out of the producing GEMM's epilogue,
    normalisation in the consuming GEMM's) on a model with massive-activation channels and large-mean
    rows: folded and unfolded forwards agree, and the fold is no further from HF fp32 than the unfolded
    bf16 path is (the bf16 storage of the residual stream, not the fold, sets the error here)."""
    from vit import vit as vit_mod
    hf = _plant_outliers(hf_oracle.build_hf(arch, seed=0), kind)
    model, _ = _build(arch, torch.bfloat16, hf)
    x = hf_oracle.make_input(arch, 3)
    want = hf_oracle.hf_forward(hf, x)
    xd = x.to(DEV, torch.bfloat16)
    try:
        with torch.no_grad():
            vit_mod.set_layernorm_folding(False)
            plain = model(xd).float().cpu()
            vit_mod.set_layernorm_folding(True, mlp=True)
            folded = model(xd).float().cpu()
    finally:
        vit_mod.set_layernorm_folding(True, mlp=True)
    assert torch.isfinite(folded).all()
    e_plain = (plain - want).abs().max().item()
    e_fold = (folded - want).abs().max().item()
    # With every channel shifted by 4 .. 6 one bf16 ulp of the residual stream is 6 % of a row's spread: the two
    # launch chains round a few values differently and that noise is amplified from block to block whichever
    # way LayerNorm is computed (the kernel-level tests check the fold itself on |mean| / std up to 1000, bit
    # for bit against fp32) — so here the bar is "as close to HF fp32 as the unfolded bf16 path", not equality.
    floor = 0.9995 if kind == "massive_channels" else 0.995
    assert _cos(folded, plain) >= floor, f"cosine folded vs unfolded {_cos(folded, plain)}"
    assert _cos(folded, want) >= min(0.999, _cos(plain, want) - 5e-4), f"cosine {_cos(folded, want)} (unfolded {_cos(plain, want)})"
    assert e_fold <= 1.5 * e_plain + 0.02, f"max-abs folded {e_fold} vs unfolded {e_plain}"


def test_repack_after_data_write_needs_invalidate():
    """Writes THROUGH ``param.data`` bump no version counter: ``VIT.invalidate_packed()`` is the documented
    way to drop the packed / folded operands afterwards (ADVICE r1); the unfused path, which reads the
    parameters directly, is the witness."""
    from vit import vit as vit_mod
    model, _ = _build("tiny-b", torch.bfloat16)
    x = hf_oracle.make_input("tiny-b", 2).to(DEV, torch.bfloat16)
    with torch.no_grad():
        before = model(x).clone()
        for p_ in model.encoder.layer[0].intermediate.parameters():
            p_.data.mul_(1.7)                                  # invisible to the caches
        model.encoder.layer[1].layernorm_before.weight.data.mul_(0.5)
        model.invalidate_packed()
        after = model(x).clone()
        vit_mod.set_fused(False)
        try:
            unfused = model(x)
        finally:
            vit_mod.set_fused(True)
    assert not torch.equal(before, after)
    assert _cos(after, unfused) >= 0.9995 and (after.float() - unfused.float()).abs().max().item() <= 0.1


def test_uint8_nhwc_input_matches_hf_image_processor_path():
    """Row f4 of SURVEY.md section 8: raw uint8 NHWC pixels in, the HF ViTImageProcessor arithmetic
    (rescale 1/255, mean 0.5, std 0.5) folded into the patch-embedding kernel.  Oracle: the same
    arithmetic in fp32 on the CPU followed by HF ViTModel."""
    model, hf = _build("vit-b16-224", torch.bfloat16)
    g = torch.Generator().manual_seed(7)
    x_u8 = torch.randint(0, 256, (3, 224, 224, 3), generator=g, dtype=torch.uint8)
    pixel_values = ((x_u8.float() * (1.0 / 255.0)) - 0.5) / 0.5
    want = hf_oracle.hf_forward(hf, pixel_values.permute(0, 3, 1, 2).contiguous())
    with torch.no_grad():
        got = model.forward_uint8(x_u8.to(DEV)).float().cpu()
        ref_path = model(pixel_values.permute(0, 3, 1, 2).contiguous().to(DEV, torch.bfloat16)).float().cpu()
        pooled = model.pooled(x_u8.to(DEV)).float().cpu()
    assert torch.isfinite(got).all()
    assert _cos(got, want) >= 0.999, f"cosine {_cos(got, want)}"
    assert (got - want).abs().max().item() <= 0.15, f"max-abs {(got - want).abs().max().item()}"
    assert _cos(got, ref_path) >= 0.9995
    assert torch.equal(pooled, got[:, 0, :].bfloat16().float())


def test_pooler_head_matches_hf_pooler():
    """Row f2: HF ViTModel(add_pooling_layer=True).pooler_output == VIT(add_pooling_layer=True).pooler_output."""
    from transformers import ViTConfig, ViTModel
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    arch = "tiny-b"
    torch.manual_seed(3)
    hf = ViTModel(ViTConfig(**hf_oracle.ARCHS[arch]), add_pooling_layer=True).eval()
    with torch.no_grad():
        hf.pooler.dense.bias.copy_(torch.randn_like(hf.pooler.dense.bias) * 0.1)
    x = hf_oracle.make_input(arch, 5)
    with torch.no_grad():
        want = hf(pixel_values=x).pooler_output
    for dtype, tol in ((torch.float32, 1e-4), (torch.bfloat16, 3e-2)):
        model = VIT(**hf_oracle.vit_kwargs(arch), add_pooling_layer=True)
        transfer_pretrained_weights(hf, model, verbose=False)
        model = model.to(DEV, dtype).eval()
        with torch.no_grad():
            got = model.pooler_output(x.to(DEV, dtype)).float().cpu()
        assert got.shape == want.shape
        assert (got - want).abs().max().item() <= tol, f"{dtype}: max-abs {(got - want).abs().max().item()}"


def test_peer_gather_matches_nccl_world2():
    """Two ranks on two GPUs: the fused pool + peer-store gather kernel returns the same bits as
    vt_pool_cls + NCCL all-gather, step after step (tests/peer_gather_worker.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import socket
    import torch.multiprocessing as mp
    import peer_gather_worker
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(peer_gather_worker.run, args=(2, port), nprocs=2, join=True)


def test_classifier_head_matches_hf_image_classification():
    """Row f2: HF ViTForImageClassification(...).logits == VIT(num_labels=...).logits, weights moved by
    transfer_pretrained_weights (source keys carry the ``vit.`` prefix, classifier.* is transposed)."""
    from transformers import ViTConfig, ViTForImageClassification
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    arch = "tiny-b"
    torch.manual_seed(5)
    hf = ViTForImageClassification(ViTConfig(**hf_oracle.ARCHS[arch], num_labels=40)).eval()
    with torch.no_grad():
        hf.classifier.weight.copy_(torch.randn_like(hf.classifier.weight) * 0.1)
        hf.classifier.bias.copy_(torch.randn_like(hf.classifier.bias) * 0.1)
    x = hf_oracle.make_input(arch, 5)
    with torch.no_grad():
        want = hf(pixel_values=x).logits
    for dtype, tol in ((torch.float32, 1e-4), (torch.bfloat16, 5e-2)):
        model = VIT(**hf_oracle.vit_kwargs(arch), num_labels=40)
        transfer_pretrained_weights(hf, model, verbose=False)
        model = model.to(DEV, dtype).eval()
        with torch.no_grad():
            got = model.logits(x.to(DEV, dtype)).float().cpu()
        assert got.shape == want.shape == (5, 40)
        assert (got - want).abs().max().item() <= tol, f"{dtype}: max-abs {(got - want).abs().max().item()}"


def test_reference_triton_forward_matches_ours(tmp_path):
    """SURVEY.md 8c / 8f-1: the reference's OWN forward (its VIT module, its Triton kernels, its loader,
    unmodified, from baseline/_ref — see oracle/fetch_reference.sh) run on this GPU in a separate process,
    compared with ours on the same weights and pixels.  Pins parity to the reference itself, not only to
    HF.  Skipped when the copy is absent or the 2024 Triton source does not run under this Triton."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.isdir(os.path.join(root, "baseline", "_ref", "vit")):
        pytest.skip("baseline/_ref/vit absent: oracle/fetch_reference.sh copies the reference package there")
    model, hf = _build("vit-b16-224", torch.float32)
    x = hf_oracle.make_input("vit-b16-224", 2)
    src, dst = str(tmp_path / "in.pt"), str(tmp_path / "out.pt")
    torch.save({"state_dict": hf.state_dict(), "input": x}, src)
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    proc = subprocess.run([sys.executable, os.path.join(root, "tools", "run_reference_triton.py"), src, dst],
                          env=env, capture_output=True, text=True, timeout=1500)
    assert os.path.exists(dst), proc.stdout[-2000:] + proc.stderr[-2000:]
    res = torch.load(dst)
    if res["error"] is not None:
        pytest.skip("the reference did not run on this box: " + res["error"].strip().splitlines()[-1])
    ref = res["output"]
    want = hf_oracle.hf_forward(hf, x)
    with torch.no_grad():
        ours32 = model(x.to(DEV)).cpu()
        ours16 = model.to(torch.bfloat16)(x.to(DEV, torch.bfloat16)).float().cpu()
    # the reference multiplies in TF32 (tl.dot allow_tf32, matmul.py:92): ~3e-3 from HF fp32 (SURVEY.md 7.2)
    assert (ref - want).abs().max().item() <= 2e-2, f"reference vs HF {(ref - want).abs().max().item()}"
    assert (ours32 - ref).abs().max().item() <= 2e-2, f"ours fp32 vs reference {(ours32 - ref).abs().max().item()}"
    assert (ours32 - want).abs().max().item() <= (ref - want).abs().max().item() + 1e-3     # at least as close to HF
    assert _cos(ours16, ref) >= 0.999 and (ours16 - ref).abs().max().item() <= 0.15


@pytest.mark.parametrize("arch", ["tiny-b", "vit-b16-224"])
def test_fp8_path_parity_vs_hf(arch):
    """SURVEY.md 8f-3: QKV / fc1 / fc2 on e4m3 operands (tcgen05.mma kind::f8f6f4), off by default.  Stated parity
    against HF fp32 on random-init weights: cosine >= 0.995, max-abs <= 0.5 on the final hidden states
    (bf16 path: >= 0.999 / <= 0.15); the measured values are printed."""
    from vit import vit as vit_mod
    model, hf = _build(arch, torch.bfloat16)
    x = hf_oracle.make_input(arch, 3)
    want = hf_oracle.hf_forward(hf, x)
    xd = x.to(DEV, torch.bfloat16)
    try:
        with torch.no_grad():
            bf16 = model(xd).float().cpu()
            vit_mod.set_fp8(True)
            fp8 = model(xd).float().cpu()
            assert torch.equal(fp8, model(xd).float().cpu())
    finally:
        vit_mod.set_fp8(False)
    assert torch.isfinite(fp8).all() and not torch.equal(fp8, bf16)
    cos, err = _cos(fp8, want), (fp8 - want).abs().max().item()
    print(f"fp8 {arch}: cosine {cos:.6f} max-abs {err:.4f} (bf16 path: {_cos(bf16, want):.6f} / {(bf16 - want).abs().max().item():.4f})")
    assert cos >= 0.995 and err <= 0.5, f"cosine {cos}, max-abs {err}"


def _wide_model(dim, layers=2, seed=0):
    """A VIT of width `dim` (64-wide heads, 32x32 images, 16-pixel patches) with the oracle's initialisation:
    weights 0.02 randn, biases 0.02 randn, LayerNorm gamma 1 + 0.02 randn."""
    from vit.vit import VIT
    model = VIT(height=32, width=32, channels=3, patch_size=16, hidden_dim=dim, num_heads=dim // 64,
                num_layers=layers, mlp_dim=4 * dim)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            noise = 0.02 * torch.randn(p.shape, generator=g)
            p.copy_(1.0 + noise if "layernorm" in name and name.endswith("weight") else noise)
    return model.to(DEV, torch.bfloat16).eval()


def _fp8_and_bf16(model, x):
    from vit import vit as vit_mod
    try:
        with torch.no_grad():
            bf16 = model(x).float().cpu()
            vit_mod.set_fp8(True)
            fp8 = model(x).float().cpu()
    finally:
        vit_mod.set_fp8(False)
    return fp8, bf16


def test_fp8_path_at_width_1664():
    """D = 1664 (ViT-bigG's width): vt_layernorm_fp8 runs at 7 vectors per lane; the FP8 forward meets the FP8 gate
    (cosine >= 0.995, max-abs <= 0.5) against the bf16 forward of the same model."""
    model = _wide_model(1664)
    x = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(1)).to(DEV, torch.bfloat16)
    fp8, bf16 = _fp8_and_bf16(model, x)
    assert torch.isfinite(fp8).all() and not torch.equal(fp8, bf16)
    cos, err = _cos(fp8, bf16), (fp8 - bf16).abs().max().item()
    assert cos >= 0.995 and err <= 0.5, f"cosine {cos}, max-abs {err}"


def test_fp8_path_above_width_2048_takes_the_bf16_path():
    """D > 2048 has no e4m3 LayerNorm: set_fp8(True) runs the bf16 forward, bit for bit."""
    model = _wide_model(2176)
    x = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(2)).to(DEV, torch.bfloat16)
    fp8, bf16 = _fp8_and_bf16(model, x)
    assert torch.equal(fp8, bf16)
