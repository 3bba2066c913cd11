"""Model factories under the reference's registry names (egom2p/models/egom2p_model.py:982-1123) plus `create_model`
(egom2p/utils/timm/model_builder.py:27-74). `register_into_reference()` re-registers them in the reference's own timm
registry so `run_training_egom2p.py --model egom2p_base_12e_12d_swiglu_nobias` builds the B200 module unchanged
(later registrations override earlier ones, egom2p/utils/timm/registry.py:39)."""
from __future__ import annotations

from functools import partial
from typing import Callable, Dict

from torch import nn

from .model import EgoM2P, LayerNorm

_ENTRYPOINTS: Dict[str, Callable] = {}


def register_model(fn):
    _ENTRYPOINTS[fn.__name__] = fn
    return fn


def _swiglu(depth_e, depth_d, dim, heads, causal=False):
    def build(encoder_embeddings, decoder_embeddings, **kwargs):
        return EgoM2P(encoder_embeddings=encoder_embeddings, decoder_embeddings=decoder_embeddings, encoder_depth=depth_e,
                      decoder_depth=depth_d, dim=dim, num_heads=heads, mlp_ratio=4, qkv_bias=False, proj_bias=False,
                      mlp_bias=False, norm_layer=partial(LayerNorm, eps=1e-6, bias=False), act_layer=nn.SiLU, gated_mlp=True,
                      decoder_causal_mask=causal, **kwargs)
    return build


for _name, _args in {
    "egom2p_tiny_6e_6d_swiglu_nobias": (6, 6, 384, 6),
    "egom2p_small_8e_8d_swiglu_nobias": (8, 8, 512, 8),
    "egom2p_base_12e_12d_swiglu_nobias": (12, 12, 768, 12),
    "egom2p_base_12e_12d_swiglu_nobias_causal": (12, 12, 768, 12, True),
}.items():
    _fn = _swiglu(*_args)
    _fn.__name__ = _name
    register_model(_fn)


def _gelu(depth_e, depth_d, dim, heads):
    """The GELU / bias family with the arguments the reference passes (4M's fm_*_gelu renamed fm_ -> egom2p_): biases on
    every Linear and LayerNorm, nn.GELU MLP, everything else at the constructor defaults."""
    def build(encoder_embeddings, decoder_embeddings, **kwargs):
        return EgoM2P(encoder_embeddings=encoder_embeddings, decoder_embeddings=decoder_embeddings, encoder_depth=depth_e,
                      decoder_depth=depth_d, dim=dim, num_heads=heads, mlp_ratio=4, qkv_bias=True,
                      norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)
    return build


for _name, _args in {
    "egom2p_tiny_6e_6d_gelu": (6, 6, 384, 6),
    "egom2p_small_8e_8d_gelu": (8, 8, 512, 8),
    "egom2p_base_12e_12d_gelu": (12, 12, 768, 12),
}.items():
    _fn = _gelu(*_args)
    _fn.__name__ = _name
    register_model(_fn)


def model_entrypoint(name: str) -> Callable:
    return _ENTRYPOINTS[name]


def is_model(name: str) -> bool:
    return name in _ENTRYPOINTS


def create_model(model_name: str, pretrained: bool = False, **kwargs):
    if pretrained:
        raise NotImplementedError("no checkpoints are reachable offline; load a state_dict explicitly")
    if not is_model(model_name):
        raise RuntimeError("Unknown model (%s)" % model_name)
    kwargs = {k: v for k, v in kwargs.items() if v is not None}
    return model_entrypoint(model_name)(**kwargs)


def register_into_reference() -> None:
    """Override the same-named entries of the reference registry (needs the reference package importable)."""
    from egom2p.utils.timm import registry as ref_registry  # type: ignore
    for name, fn in _ENTRYPOINTS.items():
        fn.__module__ = "egom2p_b200.registry"
        ref_registry._model_entrypoints[name] = fn
