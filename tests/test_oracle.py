"""CPU: the oracle restatement is pinned against HuggingFace ViTModel (live and committed golden
outputs), and the loader against digests produced by the reference's own loader."""
import hashlib
import json
import os

import pytest
import torch

from oracle import hf_oracle, restatement
from vit.utils import transfer_pretrained_weights
from vit.vit import VIT


def _custom_state_dict(arch, hf_model=None):
    model = VIT(**hf_oracle.vit_kwargs(arch))
    if hf_model is None:
        hf_model = hf_oracle.build_hf(arch, seed=0)
    transfer_pretrained_weights(hf_model, model, verbose=False)
    return model.state_dict(), hf_model


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_restatement_matches_golden_hf(arch, golden_dir):
    gold = torch.load(os.path.join(golden_dir, f"hf_{arch}.pt"))
    sd, hf = _custom_state_dict(arch, hf_model=hf_oracle.build_hf_golden(gold))
    x = hf_oracle.golden_input(gold)
    # the stored HF output is reproduced by HF itself here (pins transformers/torch numerics)
    live = hf_oracle.hf_forward(hf, x)
    assert torch.allclose(live, gold["output"], atol=1e-5, rtol=0)
    out = restatement.vit_forward(sd, x)
    assert out.shape == gold["output"].shape
    assert (out - gold["output"]).abs().max().item() <= 2e-5


def test_restatement_matches_hf_vit_b16(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "hf_vit-b16-224.pt"))
    sd, hf = _custom_state_dict("vit-b16-224")
    x = hf_oracle.make_input("vit-b16-224", gold["batch"], seed=gold["input_seed"])
    live = hf_oracle.hf_forward(hf, x)
    out = restatement.vit_forward(sd, x)
    assert (out - live).abs().max().item() <= 2e-5
    if str(torch.__version__) == gold["torch"]:
        assert (live[:, gold["tokens"]] - gold["output"]).abs().max().item() <= 1e-5


def test_restatement_edge_batch_sizes():
    sd, hf = _custom_state_dict("tiny-b")
    for b in (1, 2):
        x = hf_oracle.make_input("tiny-b", b, seed=7)
        assert (restatement.vit_forward(sd, x) - hf_oracle.hf_forward(hf, x)).abs().max().item() <= 2e-5
    empty = restatement.vit_forward(sd, hf_oracle.make_input("tiny-b", 0))
    assert empty.shape == (0, 17, 128)


def _digest(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def test_loader_matches_reference_loader_digests(golden_dir):
    """transfer_pretrained_weights == the reference's own loader, tensor by tensor (990 keys)."""
    with open(os.path.join(golden_dir, "loader_vit-b16-224.json")) as f:
        gold = json.load(f)
    hf = hf_oracle.build_hf("vit-b16-224", seed=0)
    src = {k: _digest(v) for k, v in hf.state_dict().items()}
    if src != gold["source"]:
        pytest.skip(f"HF random init differs from the fixture's (torch {torch.__version__} vs {gold['torch']})")
    sd, _ = _custom_state_dict("vit-b16-224", hf_model=hf)
    assert len(sd) == 990 == len(gold["custom"])
    assert {k: _digest(v) for k, v in sd.items()} == gold["custom"]


@pytest.mark.parametrize("arch,layers,heads,dh", [("tiny-b", 2, 2, 64), ("tiny-h", 2, 2, 80)])
def test_loader_slices(arch, layers, heads, dh):
    sd, hf = _custom_state_dict(arch)
    hsd = hf.state_dict()
    for l in range(layers):
        for proj in ("query", "key", "value"):
            W = hsd[f"encoder.layer.{l}.attention.attention.{proj}.weight"]
            b = hsd[f"encoder.layer.{l}.attention.attention.{proj}.bias"]
            for h in range(heads):
                assert torch.equal(sd[f"encoder.layer.{l}.attention.attention.{h}.{proj}.weight"], W.T[:, h * dh:(h + 1) * dh])
                assert torch.equal(sd[f"encoder.layer.{l}.attention.attention.{h}.{proj}.bias"], b[h * dh:(h + 1) * dh])
        assert torch.equal(sd[f"encoder.layer.{l}.intermediate.weight"], hsd[f"encoder.layer.{l}.intermediate.dense.weight"].T)
        assert torch.equal(sd[f"encoder.layer.{l}.attention.output.weight"], hsd[f"encoder.layer.{l}.attention.output.dense.weight"].T)
    assert torch.equal(sd["embeddings.projection.weight"], hsd["embeddings.patch_embeddings.projection.weight"])
