"""Host-side utilities with the reference's names (vit/utils.py): weight transfer from a HuggingFace
``ViTModel``, CUDA-graph capture of a forward, and a two-model latency benchmark."""
import functools
import logging
import re
from typing import List, Tuple

import numpy as np
import torch

from .load_weights import map_attn_layers, map_non_attn_layers

logger = logging.getLogger("vit_b200")


def tensor_info(func_name):
    """Decorator logging the shapes of tensor arguments / results (reference utils.py:18-42)."""
    def decorator(func):
        @functools.wraps(func)
        def wrapper(*args, **kwargs):
            shapes_in = [tuple(a.shape) for a in list(args) + list(kwargs.values()) if isinstance(a, torch.Tensor)]
            logger.info("%s called with %s", func_name, shapes_in)
            results = func(*args, **kwargs)
            outs = results if isinstance(results, (tuple, list)) else (results,)
            logger.info("%s returned %s", func_name, [tuple(r.shape) for r in outs if isinstance(r, torch.Tensor)])
            return results
        return wrapper
    return decorator


def _dense_mapping(num_layers: int) -> dict:
    mapping = {
        'embeddings.cls_token': 'embeddings.cls_token',
        'embeddings.position_embeddings': 'embeddings.position_embeddings',
        'embeddings.patch_embeddings.projection.weight': 'embeddings.projection.weight',
        'embeddings.patch_embeddings.projection.bias': 'embeddings.projection.bias',
        'layernorm.weight': 'layernorm.weight',
        'layernorm.bias': 'layernorm.bias',
        'pooler.dense.weight': 'pooler.dense.weight',
        'pooler.dense.bias': 'pooler.dense.bias',
        'classifier.weight': 'classifier.weight',     # ViTForImageClassification head, VIT(num_labels=...)
        'classifier.bias': 'classifier.bias',
        'embeddings.mask_token': 'embeddings.mask_token',   # ViTModel(use_mask_token=True), VIT(use_mask_token=True)
        'decoder.0.weight': 'decoder.0.weight',             # ViTForMaskedImageModeling, VIT(add_decoder=True)
        'decoder.0.bias': 'decoder.0.bias',
    }
    for i in range(num_layers):
        pre = f'encoder.layer.{i}.'
        for hf, ours in (('output.dense', 'output'), ('intermediate.dense', 'intermediate'),
                         ('attention.output.dense', 'attention.output'),
                         ('layernorm_before', 'layernorm_before'), ('layernorm_after', 'layernorm_after')):
            for kind in ('weight', 'bias'):
                mapping[f'{pre}{hf}.{kind}'] = f'{pre}{ours}.{kind}'
    return mapping


_HF_QKV = re.compile(r"^encoder\.layer\.(\d+)\.attention\.attention\.(query|key|value)\.(weight|bias)$")


def transfer_pretrained_weights(pretrained_model: torch.nn.Module, custom_model: torch.nn.Module,
                                verbose: bool = True) -> torch.nn.Module:
    """Copy every weight of a HuggingFace ``ViTModel`` into ``custom_model`` (a ``vit.vit.VIT``).

    Same call and result as the reference (utils.py:45-113); the layer count comes from the models.
    Keys of the source may carry a ``vit.`` prefix (``ViTForImageClassification``, ``ViTForMaskedImageModeling``).
    """
    source = {(k[4:] if k.startswith('vit.') else k): v for k, v in pretrained_model.state_dict().items()}
    dest = custom_model.state_dict()

    layer_ids = [int(m.group(1)) for m in map(_HF_QKV.match, source) if m]
    num_layers = (max(layer_ids) + 1) if layer_ids else 0

    for name, tensor in source.items():
        m = _HF_QKV.match(name)
        if m:
            dest = map_attn_layers(m.group(1), m.group(2), m.group(3), tensor, dest)
    dest = map_non_attn_layers(source_state_dict=source, dest_state_dict=dest,
                               weight_mapping=_dense_mapping(num_layers))

    custom_model.load_state_dict(dest, strict=False)

    if verbose:
        untouched = [k for k, v in custom_model.state_dict().items() if torch.all(v == 0)]
        if untouched:
            # HF zero-initialises biases, so a randomly initialised source lists every bias here.
            print(f"Some layer are not initialized: {untouched}")
    return custom_model


def capture_cuda_graph(model, static_input):
    """Warm up on a side stream, then capture one forward into a CUDA graph (reference
    utils.py:115-133).  Returns (graph, static_output); replay with ``graph.replay()`` after copying
    new data into ``static_input``."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.no_grad(), torch.cuda.stream(side):
        for _ in range(3):
            model(static_input)
    torch.cuda.current_stream().wait_stream(side)

    graph = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(graph):
        static_output = model(static_input)
    return graph, static_output


def timed(fn, input):
    """Run ``fn(input)`` and return (result, milliseconds) using CUDA events on the current stream."""
    start = torch.cuda.Event(enable_timing=True)
    end = torch.cuda.Event(enable_timing=True)
    start.record()
    result = fn(input)
    end.record()
    torch.cuda.synchronize()
    return result, start.elapsed_time(end)


def _last_hidden(out):
    if isinstance(out, torch.Tensor):
        return out
    if hasattr(out, 'last_hidden_state'):
        return out.last_hidden_state
    return out[0]


def benchmark(model1: torch.nn.Module, model2: torch.nn.Module,
              input_shape: Tuple[int, int, int] = (3, 224, 224),
              batch_sizes: List[int] = [1, 4, 16, 32, 64, 128, 256],
              warmups: int = 25, reps: int = 100):
    """Median forward latency (ms) of two models per batch size (reference utils.py:136-178).
    Yields (batch_size, model1_ms, model2_ms); logs the mean absolute output difference."""
    p = next(model1.parameters())
    for bs in batch_sizes:
        a = torch.randn((bs, *input_shape)).to(device=p.device, dtype=p.dtype)
        with torch.no_grad():
            for _ in range(warmups):
                model1(a)
                model2(a)
            t1 = [timed(model1, a) for _ in range(reps)]
            t2 = [timed(model2, a) for _ in range(reps)]
        o1, o2 = _last_hidden(t1[-1][0]), _last_hidden(t2[-1][0])
        logger.info("batch %d: mean |diff| %.3e", bs, torch.mean(torch.abs(o1.float() - o2.float())).item())
        yield (bs, round(float(np.median([t for _, t in t1])), 2), round(float(np.median([t for _, t in t2])), 2))
