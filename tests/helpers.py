"""Shared helpers for the parity tests: tiny/full configs that mirror tests/golden/make_golden.py."""
import os

import numpy as np
import torch

from must3r_b200 import synthetic as syn
from oracle import must3r_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

TINY_ENC = orc.EncoderConfig(img_size=(64, 64), embed_dim=128, depth=2, num_heads=2)
TINY_DEC = orc.DecoderConfig(img_size=(64, 64), enc_embed_dim=128, embed_dim=128, depth=3, num_heads=2)


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name))


def tiny_oracle(seed=7, enc_over=None, dec_over=None):
    import dataclasses
    ecfg = dataclasses.replace(TINY_ENC, **(enc_over or {}))
    dcfg = dataclasses.replace(TINY_DEC, **(dec_over or {}))
    esd = syn.encoder_state_dict(seed, embed_dim=ecfg.embed_dim, depth=ecfg.depth)
    dsd = syn.decoder_state_dict(seed, enc_embed_dim=dcfg.enc_embed_dim, embed_dim=dcfg.embed_dim,
                                 depth=dcfg.depth, output_dim=dcfg.output_dim, feedback_type=dcfg.feedback_type)
    return orc.OracleEncoder(esd, ecfg), orc.OracleDecoder(dsd, dcfg)


def full_oracle(size, seed=0):
    ecfg = orc.EncoderConfig(img_size=(size, size))
    dcfg = orc.DecoderConfig(img_size=(size, size))
    return (orc.OracleEncoder(syn.encoder_state_dict(seed), ecfg),
            orc.OracleDecoder(syn.decoder_state_dict(seed), dcfg))


def digest(t, max_elems=4096):  # same sampling as tests/golden/make_golden.py
    f = t.detach().float().flatten().cpu()
    step = max(1, f.numel() // max_elems)
    return np.concatenate([f[::step][:max_elems].numpy(),
                           np.array([f.mean(), f.std(), f.abs().sum() / f.numel()], dtype=np.float32)])


def keyframe_frame(seed, H=48, W=64, shift=0.0):
    """A random postprocessed frame (pts3d, pts3d_local with positive depth, conf >= 1) for the keyframe overlap tests."""
    g = torch.Generator().manual_seed(seed)
    pts = torch.randn(1, 1, H, W, 3, generator=g) * 2.0 + shift
    loc = pts.clone()
    loc[..., 2] = loc[..., 2].abs() + 1.0
    conf = 1.0 + torch.rand(1, 1, H, W, generator=g) * 3.0
    return {"pts3d": pts, "pts3d_local": loc, "conf": conf}


KEYFRAME_METHODS = ["kdtree-scipy", "quadrant_x2-kdtree-scipy", "quadrant_x4-kdtree-scipy"]
KEYFRAME_DB = [(10 + i, 0.5 * i) for i in range(3)]      # (seed, shift) of the three keyframes stored in the database
KEYFRAME_QUERIES = [(50, 0.2), (51, 3.0)]                 # an overlapping and a far-away frame
KEYFRAME_CAM = (0.1, -0.2, 0.3)


def rel(a, b):
    a = torch.as_tensor(np.asarray(a)).double()
    b = torch.as_tensor(np.asarray(b)).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))
