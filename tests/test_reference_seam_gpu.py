"""Operator seam A/B (SURVEY.md §8b): the must3r_b200 model against stored outputs of the UNMODIFIED reference
(tests/golden/full_model_digest.npz), the reference's RoPE as served by ``must3r_b200.compat.curope`` (-> m3r_rope_2d)
against its PyTorch fallback's arithmetic, and, where the reference is installed under oracle/_ref
(oracle/install_reference.py), the reference itself running its CUDA forward on that shim.  Reference call sites:
dust3r/croco/models/pos_embed.py:104-110 (import-time selection), curope/curope2d.py:32-39, curope.cpp:49-69."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baseline import ref_loader  # noqa: E402
from helpers import load_golden, digest, rel  # noqa: E402
from must3r_b200 import synthetic as syn  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    if not ref_loader.available():
        pytest.skip("the reference is not installed under oracle/_ref")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return ref_loader.load_reference(curope_shim=True)


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def test_reference_selected_the_shim(ref):
    """The reference picks the shim as its `curope`, and its CUDA fp32 forward on it reproduces its own CPU outputs
    (made with the PyTorch RoPE fallback)."""
    assert ref.rope_class == "cuRoPE2D"
    import curope
    assert curope.__name__ == "must3r_b200.compat.curope"
    dev = torch.device("cuda", 0)
    imgs, ts = syn.synthetic_views(3, 224, 224, seed=2)
    imgs, tsd = imgs.to(dev), ts.to(dev)
    renc = ref.Dust3rEncoder(img_size=(224, 224)).eval()
    rdec = ref.MUSt3R(img_size=(224, 224), feedback_type="single_mlp", memory_mode="kv", landscape_only=False).eval()
    renc.load_state_dict(syn.encoder_state_dict(0)); rdec.load_state_dict(syn.decoder_state_dict(0))
    renc, rdec = renc.to(dev), rdec.to(dev)
    with torch.no_grad():
        rx, rpos = renc(imgs, tsd)
        rmem, _ = rdec(rx[None, :2], rpos[None, :2], tsd[None, :2], None)
        rmem, _ = rdec(rx[None, 2:3], rpos[None, 2:3], tsd[None, 2:3], rmem)
        _, rpm = rdec(rx[None], rpos[None], tsd[None], rmem, render=True)
    g = load_golden("full_model_digest.npz")
    assert rel(digest(rx), g["224.enc_x"]) < 2e-5 and rel(digest(rpm), g["224.pm_render"]) < 5e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_shim_rope_matches_reference_fallback(dtype):
    """cuRoPE2D (the shim, called as the reference's curope2d.py:32-39 calls it) vs the reference's PyTorch RoPE2D
    semantics (pos_embed.py:111-157), restated in fp64 here."""
    from must3r_b200.compat import curope
    torch.manual_seed(0)
    B, H, N, D = 2, 3, 35, 64
    tok = torch.randn(B, H, N, D, device="cuda", dtype=dtype)
    pos = torch.stack([torch.randint(0, 24, (B, N), device="cuda"), torch.randint(0, 32, (B, N), device="cuda")], -1)
    rope = curope.cuRoPE2D(freq=100.0, F0=0.4375)
    want = tok.clone().double()
    Q = D // 4
    inv = 0.4375 / (100.0 ** (torch.arange(Q, device="cuda", dtype=torch.float64) / Q))
    for axis in range(2):
        ang = pos[..., axis].double()[:, None, :, None] * inv                      # [B,1,N,Q]
        c, s = ang.cos(), ang.sin()
        u = want[..., axis * 2 * Q: axis * 2 * Q + Q].clone()
        v = want[..., axis * 2 * Q + Q: (axis + 1) * 2 * Q].clone()
        want[..., axis * 2 * Q: axis * 2 * Q + Q] = u * c - v * s
        want[..., axis * 2 * Q + Q: (axis + 1) * 2 * Q] = v * c + u * s
    got = rope(tok, pos)
    assert got.data_ptr() == tok.data_ptr()                                         # in place, like curope
    tol = {torch.float32: 2e-6, torch.float16: 6e-4, torch.bfloat16: 5e-3}[dtype]
    assert _rel(got, want) < tol


def test_unmodified_reference_on_shim_vs_must3r_b200():
    """Full ViT-L / ViT-B at 224x224, 3 views (init 2, update 1, render 3): our kernels with fp16 operands against the
    reference's fp32 outputs on the same weights and views (strided samples + moments, tests/golden/full_model_digest.npz).
    The reference's CUDA forward on the shim reproduces those outputs to 5e-5 (test_reference_selected_the_shim)."""
    from must3r_b200.model import Dust3rEncoder, MUSt3R, set_precision
    dev = torch.device("cuda", 0)
    g = load_golden("full_model_digest.npz")
    imgs, ts = syn.synthetic_views(3, 224, 224, seed=2)
    imgs, tsd = imgs.to(dev), ts.to(dev)
    set_precision(torch.float16)
    enc = Dust3rEncoder(img_size=(224, 224)); dec = MUSt3R(img_size=(224, 224), feedback_type="single_mlp", memory_mode="kv", landscape_only=False)
    enc.load_state_dict(syn.encoder_state_dict(0)); dec.load_state_dict(syn.decoder_state_dict(0))
    enc, dec = enc.to(dev).eval(), dec.to(dev).eval()
    x, pos = enc(imgs, tsd)
    mem, _ = dec(x[None, :2], pos[None, :2], tsd[None, :2], None)
    mem, pm_u = dec(x[None, 2:3], pos[None, 2:3], tsd[None, 2:3], mem)
    _, pm = dec(x[None], pos[None], tsd[None], mem, render=True)
    grid = torch.cartesian_prod(torch.arange(14), torch.arange(14))                 # (y, x) of the 14x14 patches
    assert np.array_equal(pos.cpu().numpy(), grid[None].expand(3, -1, -1).numpy())
    assert rel(digest(x), g["224.enc_x"]) < 1.2e-3 and rel(digest(pm_u), g["224.pm_upd"]) < 1.2e-3
    assert rel(digest(pm), g["224.pm_render"]) < 1.2e-3
    assert rel(digest(mem[0][11].float()), g["224.mem11"]) < 1.5e-3


def test_attention_toggle_exports():
    """must3r/model/blocks/attention.py:5-27 names exist and behave (flag only: one backend)."""
    from must3r_b200.compat import attention as att
    assert att.has_xformers is False
    att.toggle_memory_efficient_attention(True)
    assert att.is_memory_efficient_attention_enabled()
    att.toggle_memory_efficient_attention(False)
    assert not att.is_memory_efficient_attention_enabled()
    torch.manual_seed(1)
    q, k, v = (torch.randn(2, 12, 200, 64, device="cuda", dtype=torch.float16) for _ in range(3))
    out = att.attention(q, k, v)
    want = torch.nn.functional.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2).reshape(2, 200, 768)
    assert _rel(out.float(), want) < 2e-3
