"""TEST INFRASTRUCTURE — regenerates tests/golden/* (run in the build container, not on the GPU box).

    python oracle/make_golden.py

Fixtures:
  loader_vit-b16-224.json   sha256 of every tensor the REFERENCE'S OWN loader
                            (/root/reference/vit/utils.py:45-113, imported and executed here on CPU)
                            produces from the seed-0 HF ViT-B/16 model, plus digests of the source.
  hf_tiny-b.pt, hf_tiny-h.pt   sha256 of every HF weight and of the input + HF fp32 last_hidden_state for the
                            tiny archs (weights and input are regenerated from the seeds at test time and checked).
  hf_vit-b16-224.pt         HF fp32 last_hidden_state for 2 seeded images of the seed-0 ViT-B/16, CLS + 15
                            seeded patch tokens (weights are regenerated from the seed at test time: 343 MB otherwise).
"""
import contextlib
import io
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import hf_oracle  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')


digest = hf_oracle.digest


def reference_loader_digests():
    """Run the reference's transfer_pretrained_weights (needs /root/reference; CPU only)."""
    sys.path.insert(0, '/root/reference')
    for k in [k for k in sys.modules if k == 'vit' or k.startswith('vit.')]:
        del sys.modules[k]
    from vit.utils import transfer_pretrained_weights as ref_transfer
    from vit.vit import VIT as RefVIT
    hf = hf_oracle.build_hf('vit-b16-224', seed=0)
    ref_model = RefVIT(224, 224, 3, 16, 768, 12, 12)
    with contextlib.redirect_stdout(io.StringIO()):
        ref_transfer(hf, ref_model)
    out = {
        'source': {k: digest(v) for k, v in hf.state_dict().items()},
        'custom': {k: digest(v) for k, v in ref_model.state_dict().items()},
        'torch': str(torch.__version__),
    }
    sys.path.remove('/root/reference')
    for k in [k for k in sys.modules if k == 'vit' or k.startswith('vit.')]:
        del sys.modules[k]
    return out


def write_hf_fixtures(gold_dir=GOLD):
    """Fixtures of a few ten KB: weights and pixels are stored as sha256 digests (hf_oracle.build_hf_golden
    and hf_oracle.golden_input rebuild them from the seeds and check them), and of the ViT-B/16 output only the
    CLS token and a seeded sample of 15 patch tokens are kept."""
    os.makedirs(gold_dir, exist_ok=True)
    for arch, batch in (('tiny-b', 3), ('tiny-h', 3)):
        hf = hf_oracle.build_hf(arch, seed=0)
        x = hf_oracle.make_input(arch, batch)
        y = hf_oracle.hf_forward(hf, x)
        torch.save({'arch': arch, 'model_seed': 0, 'input_seed': 1234, 'batch': batch,
                    'state_dict_sha256': {k: digest(v) for k, v in hf.state_dict().items()},
                    'input_digest': digest(x), 'output': y, 'torch': str(torch.__version__)},
                   os.path.join(gold_dir, f'hf_{arch}.pt'))

    hf = hf_oracle.build_hf('vit-b16-224', seed=0)
    x = hf_oracle.make_input('vit-b16-224', 2)
    y = hf_oracle.hf_forward(hf, x)
    n_tok = y.shape[1]
    sample = torch.randperm(n_tok - 1, generator=torch.Generator().manual_seed(0))[:15] + 1
    tokens = torch.cat([torch.zeros(1, dtype=torch.long), sample.sort().values])
    torch.save({'arch': 'vit-b16-224', 'model_seed': 0, 'input_seed': 1234, 'batch': 2, 'tokens': tokens,
                'output': y[:, tokens].clone(), 'input_digest': digest(x), 'torch': str(torch.__version__)},
               os.path.join(gold_dir, 'hf_vit-b16-224.pt'))


def main():
    os.makedirs(GOLD, exist_ok=True)
    with open(os.path.join(GOLD, 'loader_vit-b16-224.json'), 'w') as f:
        json.dump(reference_loader_digests(), f, indent=0, sort_keys=True)
    write_hf_fixtures()
    print('golden fixtures written to', GOLD)


if __name__ == '__main__':
    main()
