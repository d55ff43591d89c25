"""Shared helpers for the test tiers."""
import copy
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_CACHE = {}

# Decoded-image source sizes (h, w) the GPU resize is checked at, against Pillow and the oracle's restatement
RESIZE_SOURCES = [
    (200, 200), (300, 260), (97, 131),
    (224, 300), (300, 224), (224, 97), (97, 224),      # one axis only: the horizontal pass alone writes the output, or
                                                       # the vertical pass alone reads the caller's buffer
    (223, 225), (225, 223),                            # near identity
    (1, 1), (1, 224), (224, 1), (2, 3), (7, 5),        # tiny sources
    (17, 600), (600, 17),                              # upscale one axis, downscale the other
    (1080, 1920), (3000, 4000),                        # strong downscales: up to 2 * ceil(src / 224) + 1 taps
]


def cached_quantized(widths):
    """Converted INT8 module for `widths` (PTQ takes a few seconds; share it across tests)."""
    from oracle import model_factory as mf
    key = ("q", tuple(widths))
    if key not in _CACHE:
        _CACHE[key] = mf.static_quantize_fbgemm(mf.make_student(widths))
    return _CACHE[key]


def with_nonzero_zero_points(gm):
    """Copy of the converted ResNet ``gm`` whose zero points are moved away from 0: block ``i``'s conv1 (ConvReLU2d, so
    its outputs clamp at the zero point) gets 3 + 2i, its output (the add_relu) 5 + 3i.  The converted ResNet never has
    a non-zero zero point on a conv input (every one is post-ReLU); after this every conv except the stem reads one.
    The module itself is edited, so the oracle (``extract_qnet``), the engine (``from_converted``) and the live fbgemm
    module all read the same definition."""
    import torch
    g = copy.deepcopy(gm)
    mods = dict(g.named_modules())
    for i in range(8):
        li, bj = i // 2 + 1, i % 2
        mods[f"layer{li}.{bj}.conv1"].zero_point = 3 + 2 * i
        name = f"layer{li}_{bj}_relu_zero_point_0"
        old = getattr(g, name)
        setattr(g, name, torch.tensor(5 + 3 * i, dtype=old.dtype) if isinstance(old, torch.Tensor) else 5 + 3 * i)
    return g
