"""Named ViT architectures (HF ``ViTConfig`` fields) and the matching ``VIT`` constructor arguments.

Product-side table: ``bench.py`` and the developer tools build models from it; the oracle under
``/oracle`` (test infrastructure) re-exports it so that the HF models it builds have the same shapes.
"""

ARCHS = {
    # name: hidden, layers, heads, mlp, patch, image
    'vit-b16-224': dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, patch_size=16, image_size=224),
    'vit-b16-384': dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, patch_size=16, image_size=384),
    'vit-l16-224': dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096, patch_size=16, image_size=224),
    'vit-h14-224': dict(hidden_size=1280, num_hidden_layers=32, num_attention_heads=16, intermediate_size=5120, patch_size=14, image_size=224),
    # small shapes with the same structure (dh 64 / dh 80 + 14-pixel patches) for fast CPU tests
    'tiny-b': dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512, patch_size=16, image_size=64),
    'tiny-h': dict(hidden_size=160, num_hidden_layers=2, num_attention_heads=2, intermediate_size=640, patch_size=14, image_size=56),
    # 12 layers x 64-wide heads: the only shape the reference's own loader handles (utils.py:53, load_weights.py:29)
    'tiny-ref': dict(hidden_size=64, num_hidden_layers=12, num_attention_heads=1, intermediate_size=256, patch_size=16, image_size=32),
}


def vit_kwargs(arch: str) -> dict:
    """Constructor arguments of vit.vit.VIT for an architecture."""
    a = ARCHS[arch]
    return dict(height=a['image_size'], width=a['image_size'], channels=3, patch_size=a['patch_size'],
                hidden_dim=a['hidden_size'], num_heads=a['num_attention_heads'],
                num_layers=a['num_hidden_layers'], mlp_dim=a['intermediate_size'])


# CLIP image encoders (HF ``CLIPVisionConfig`` fields; the OpenAI checkpoints use quick GELU, CLIP's LayerNorm eps is
# 1e-5) and the tiny shapes their tests use.  Kept apart from ARCHS: the ViT tables and tools do not see them.
CLIP_ARCHS = {
    'clip-b32-224': dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                         patch_size=32, image_size=224, projection_dim=512, hidden_act='quick_gelu'),
    'clip-b16-224': dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                         patch_size=16, image_size=224, projection_dim=512, hidden_act='quick_gelu'),
    'clip-l14-224': dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                         patch_size=14, image_size=224, projection_dim=768, hidden_act='quick_gelu'),
    'clip-l14-336': dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                         patch_size=14, image_size=336, projection_dim=768, hidden_act='quick_gelu'),
    # small shapes: 16 / 14 / 32-pixel patches, head dim 64 and 80, and a width that is no multiple of 128 (no fold)
    'tiny-clip-b16': dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                          patch_size=16, image_size=64, projection_dim=64, hidden_act='quick_gelu'),
    'tiny-clip-h14': dict(hidden_size=160, num_hidden_layers=2, num_attention_heads=2, intermediate_size=640,
                          patch_size=14, image_size=56, projection_dim=96, hidden_act='gelu'),
    'tiny-clip-b32': dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=1024,
                          patch_size=32, image_size=96, projection_dim=128, hidden_act='quick_gelu'),
}
CLIP_LAYER_NORM_EPS = 1e-5


def clip_kwargs(arch: str) -> dict:
    """Constructor arguments of vit.vit.VIT for a CLIP image encoder (``clip=True`` with its projection)."""
    a = CLIP_ARCHS[arch]
    return dict(height=a['image_size'], width=a['image_size'], channels=3, patch_size=a['patch_size'],
                hidden_dim=a['hidden_size'], num_heads=a['num_attention_heads'], num_layers=a['num_hidden_layers'],
                mlp_dim=a['intermediate_size'], hidden_act=a['hidden_act'], layer_norm_eps=CLIP_LAYER_NORM_EPS,
                clip=True, projection_dim=a['projection_dim'])
