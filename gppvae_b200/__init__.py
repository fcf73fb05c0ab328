"""gppvae_b200 -- B200 (sm_100a) implementation of GPPVAE's low-rank GP prior term.

Drop-in for the reference's `gp.GP` and `vmod.Vmodel` (ahmerb/GPPVAE, pysrc/faceplace); see DESIGN.md.
All numerics run in libgppvae_b200.so (hand-written CUDA, C ABI in include/gppvae_b200.h); there is no
CPU path: tensors must live on a CUDA device.
"""
from .gp import GP, EffectsFactor, KhatriRaoFactor, LazyEffectVb, LazyVb, LowRankFactor  # noqa: F401
from .vmod import KhatriRao, ObjectEffect, ViewEffect, Vmodel, normalize_rows  # noqa: F401

__all__ = ["GP", "Vmodel", "normalize_rows", "LowRankFactor", "KhatriRao", "KhatriRaoFactor", "LazyVb", "ObjectEffect",
           "ViewEffect", "EffectsFactor", "LazyEffectVb"]
