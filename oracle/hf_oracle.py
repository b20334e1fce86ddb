"""TEST INFRASTRUCTURE — HuggingFace ``ViTModel`` as the numeric oracle (BASELINE.json north_star).

Random-init models of the named architectures (no network, no pretrained weights), deterministic
from seeds; biases and LayerNorm affines are re-randomised because HF zero/one-initialises them
(modeling_vit.py ``_init_weights``), which would hide bias and affine bugs.
"""
import torch

import hashlib
import os
import sys

_PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "vit.triton_b200")
if _PKG not in sys.path:
    sys.path.insert(0, _PKG)
from vit.configs import ARCHS, vit_kwargs  # noqa: E402,F401  (one table for the product and its checker)


def build_hf(arch: str, seed: int = 0, randomize_affine: bool = True):
    from transformers import ViTConfig, ViTModel
    cfg = ViTConfig(**ARCHS[arch])
    torch.manual_seed(seed)
    model = ViTModel(cfg, add_pooling_layer=False).eval()
    if randomize_affine:
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith('.bias'):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.02)
                elif 'layernorm' in name and name.endswith('.weight'):
                    p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
    return model


def make_input(arch: str, batch: int, seed: int = 1234) -> torch.Tensor:
    s = ARCHS[arch]['image_size']
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, s, s), generator=g)


@torch.no_grad()
def hf_forward(model, x: torch.Tensor) -> torch.Tensor:
    return model(pixel_values=x).last_hidden_state


def digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def build_hf_golden(gold: dict):
    """The model a tests/golden/hf_<arch>.pt fixture was computed with: rebuilt from the fixture's seed and
    checked tensor by tensor against the sha256 digests the fixture stores in place of the weights."""
    model = build_hf(gold["arch"], seed=gold["model_seed"])
    got = {k: digest(v) for k, v in model.state_dict().items()}
    assert got == gold["state_dict_sha256"], (
        f"the seed-{gold['model_seed']} {gold['arch']} weights differ from the fixture's (torch {torch.__version__}, "
        f"fixture made with {gold['torch']}): regenerate tests/golden with oracle/make_golden.py")
    return model


def golden_input(gold: dict) -> torch.Tensor:
    """The pixels of a golden fixture, regenerated from its seed and checked against its digest."""
    x = make_input(gold["arch"], gold["batch"], seed=gold["input_seed"])
    assert digest(x) == gold["input_digest"], f"seed-{gold['input_seed']} input differs from the fixture's"
    return x
