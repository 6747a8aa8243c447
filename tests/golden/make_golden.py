#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference; it does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference ships no tests / golden vectors (SURVEY.md §4), so parity is pinned by these files:
weights and inputs come from the seeded generators in ``must3r_b200/synthetic.py`` (regenerated
identically by the tests), outputs come from the reference's own classes
(must3r/model/encoder.py:13 Dust3rEncoder, must3r/model/decoder.py:14 MUSt3R) and engine functions
(must3r/engine/inference.py) on CPU fp32 with the SDPA attention branch and the PyTorch RoPE fallback
(identical to curope in fp32 to 1.8e-7, SURVEY.md §0 fact 9).
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

# `roma` is only needed by postprocess(compute_cam=True) (engine/inference.py:38); stub it.
sys.modules.setdefault("roma", types.ModuleType("roma"))

from must3r.model import Dust3rEncoder, MUSt3R  # noqa: E402
from must3r.model.blocks.head import ActivationType  # noqa: E402
import must3r.engine.inference as ref_engine  # noqa: E402

from must3r_b200 import synthetic as syn  # noqa: E402

torch.set_grad_enabled(False)
torch.manual_seed(0)


def build_ref(enc_kw, dec_kw, seed=0):
    enc = Dust3rEncoder(**enc_kw).eval()
    dec = MUSt3R(**dec_kw).eval()
    esd = syn.encoder_state_dict(seed, embed_dim=enc_kw.get("embed_dim", 1024), depth=enc_kw.get("depth", 24))
    dsd = syn.decoder_state_dict(seed, enc_embed_dim=dec_kw.get("enc_embed_dim", 1024),
                                 embed_dim=dec_kw.get("embed_dim", 768), depth=dec_kw.get("depth", 12),
                                 output_dim=dec_kw.get("output_dim", 1792),
                                 feedback_type=dec_kw.get("feedback_type", None))
    enc.load_state_dict(esd, strict=True)   # also proves the synthetic key names/shapes are the reference's
    dec.load_state_dict(dsd, strict=True)
    return enc, dec


TINY_ENC = dict(img_size=(64, 64), patch_size=16, embed_dim=128, depth=2, num_heads=2)
TINY_DEC = dict(img_size=(64, 64), enc_embed_dim=128, embed_dim=128, depth=3, num_heads=2, output_dim=1792,
                feedback_type="single_mlp", memory_mode="kv", landscape_only=False)


def mem_arrays(prefix, mem, out):
    vals, labels, a, b, c = mem
    for l, v in enumerate(vals):
        out[f"{prefix}.mem{l}"] = v.numpy()
    out[f"{prefix}.labels"] = labels.numpy()
    out[f"{prefix}.tail"] = np.array([a, b, c], dtype=np.int64)


def tiny_model_golden():
    out = {}
    H, W = 32, 48
    for variant, (enc_over, dec_over) in {
        "kv": ({}, {}),
        "normy": ({}, dict(memory_mode="norm_y")),
        "raw": ({}, dict(memory_mode="raw")),
        "f0": (dict(pos_embed="RoPE100_224:512"), dict(pos_embed="RoPE100_224:512")),
        "nofb": ({}, dict(feedback_type=None)),
        "fblin": ({}, dict(feedback_type="single_linear")),
    }.items():
        enc, dec = build_ref({**TINY_ENC, **enc_over}, {**TINY_DEC, **dec_over}, seed=7)
        imgs, ts = syn.synthetic_views(5, H, W, seed=11)
        x, pos = enc(imgs, ts)
        out[f"{variant}.enc_x"] = x.numpy()
        out[f"{variant}.enc_pos"] = pos.numpy()
        # init with 2 views (decoder.py:280-285), update with 1, update with 2 (mask with Nm>0), render 5
        mem, pm0 = dec(x[None, 0:2], pos[None, 0:2], ts[None, 0:2], None)
        out[f"{variant}.pm_init"] = pm0.numpy()
        mem_arrays(f"{variant}.init", mem, out)
        mem, pm1 = dec(x[None, 2:3], pos[None, 2:3], ts[None, 2:3], mem)
        out[f"{variant}.pm_upd1"] = pm1.numpy()
        mem, pm2 = dec(x[None, 3:5], pos[None, 3:5], ts[None, 3:5], mem)
        out[f"{variant}.pm_upd2"] = pm2.numpy()
        mem_arrays(f"{variant}.final", mem, out)
        mem_r, pmr = dec(x[None], pos[None], ts[None], mem, render=True)
        out[f"{variant}.pm_render"] = pmr.numpy()
        assert mem_r[0][0] is mem[0][0]
    # single-image init: no own-mask (decoder.py:293), B=2 scenes
    enc, dec = build_ref(TINY_ENC, TINY_DEC, seed=7)
    imgs, ts = syn.synthetic_views(6, H, W, seed=12)
    x, pos = enc(imgs, ts)
    xb, pb, tb = x.view(2, 3, *x.shape[1:]), pos.view(2, 3, *pos.shape[1:]), ts.view(2, 3, 2)
    mem, pm = dec(xb[:, :1].contiguous(), pb[:, :1].contiguous(), tb[:, :1].contiguous(), None)
    out["b2.pm_init1"] = pm.numpy()
    mem, pm = dec(xb[:, 1:3].contiguous(), pb[:, 1:3].contiguous(), tb[:, 1:3].contiguous(), mem)
    out["b2.pm_upd2"] = pm.numpy()
    mem_arrays("b2.final", mem, out)
    _, pm = dec(xb, pb, tb, mem, render=True)
    out["b2.pm_render"] = pm.numpy()
    # list form with two aspect ratios (decoder.py:158): 32x48 landscape and 48x32 portrait
    imgs_p, ts_p = syn.synthetic_views(2, 48, 32, seed=13)
    xp, pp = enc(imgs_p, ts_p)
    imgs_l, ts_l = syn.synthetic_views(2, H, W, seed=14)
    xl, pl = enc(imgs_l, ts_l)
    mem, pms = dec([xl[None], xp[None]], [pl[None], pp[None]], [ts_l[None], ts_p[None]], None)
    out["list.pm0"], out["list.pm1"] = pms[0].numpy(), pms[1].numpy()
    mem_arrays("list.init", mem, out)
    mem2, pms = dec([xp[None, :1], xl[None, :1]], [pp[None, :1], pl[None, :1]], [ts_p[None, :1], ts_l[None, :1]], mem)
    out["list.pm2"], out["list.pm3"] = pms[0].numpy(), pms[1].numpy()
    mem_arrays("list.final", mem2, out)
    # ManyAR patch embedding: landscape-stored batch with one portrait view (dust3r/dust3r/patch_embed.py:32-70)
    enc_m, _ = build_ref({**TINY_ENC, "patch_embed": "ManyAR_PatchEmbed"}, TINY_DEC, seed=7)
    imgs_m, _ = syn.synthetic_views(3, H, W, seed=15)
    ts_m = torch.tensor([[H, W], [W, H], [H, W]], dtype=torch.int64)
    xm, pm_ = enc_m(imgs_m, ts_m)
    out["manyar.enc_x"], out["manyar.enc_pos"] = xm.numpy(), pm_.numpy()
    # postprocess (engine/inference.py:16-27)
    pp_out = ref_engine.postprocess(torch.from_numpy(out["kv.pm_render"]), ActivationType.NORM_EXP)
    # focal of postprocess(compute_cam=True) (engine/inference.py:29-35); the pose half needs roma, which is not installed
    from dust3r.post_process import estimate_focal_knowing_depth
    loc = pp_out["pts3d_local"]
    Hh, Ww = loc.shape[-3], loc.shape[-2]
    out["kv.post.focal"] = estimate_focal_knowing_depth(loc.reshape(-1, Hh, Ww, 3), torch.tensor((Ww / 2, Hh / 2)),
                                                         focal_mode="weiszfeld").numpy()
    # the same estimator on noisy pinhole pointmaps with known focals (a non-degenerate known-answer case)
    gen = torch.Generator().manual_seed(21)
    f_true = torch.tensor([40.0, 55.0, 70.0])
    vv, uu = torch.meshgrid(torch.arange(Hh, dtype=torch.float32), torch.arange(Ww, dtype=torch.float32), indexing="ij")
    z = 2.0 + torch.rand(3, Hh, Ww, generator=gen) * 3.0
    xl = (uu[None] - Ww / 2) * z / f_true.view(3, 1, 1)
    yl = (vv[None] - Hh / 2) * z / f_true.view(3, 1, 1)
    cam_pts = torch.stack([xl, yl, z], -1) + 0.01 * torch.randn(3, Hh, Ww, 3, generator=gen)
    cam_pts[0, 0, 0, 2] = 0.0                                   # a zero depth: exercises the nan_to_num branch
    out["cam.pts_local"] = cam_pts.numpy()
    out["cam.focal"] = estimate_focal_knowing_depth(cam_pts, torch.tensor((Ww / 2, Hh / 2)), focal_mode="weiszfeld").numpy()
    for k, v in pp_out.items():
        out[f"kv.post.{k}"] = v.numpy()
    np.savez_compressed(os.path.join(HERE, "tiny_model.npz"), **out)
    print("tiny_model.npz", len(out), "arrays")


def digest(t: torch.Tensor, max_elems=4096):
    """Strided sample + moments of a large tensor (keeps fixtures small)."""
    f = t.detach().float().flatten()
    step = max(1, f.numel() // max_elems)
    return np.concatenate([f[::step][:max_elems].numpy(),
                           np.array([f.mean(), f.std(), f.abs().sum() / f.numel()], dtype=np.float32)])


def full_model_golden():
    """Full-size ViT-L encoder / ViT-B decoder (the real architecture) -> digests only."""
    out = {}
    for tag, (H, W, size) in {"224": (224, 224, 224), "512": (384, 512, 512)}.items():
        enc, dec = build_ref(dict(img_size=(size, size)),
                             dict(img_size=(size, size), feedback_type="single_mlp", memory_mode="kv",
                                  landscape_only=False), seed=0)
        imgs, ts = syn.synthetic_views(3, H, W, seed=2)
        x, pos = enc(imgs, ts)
        out[f"{tag}.enc_x"] = digest(x)
        mem, pm = dec(x[None, :2], pos[None, :2], ts[None, :2], None)
        out[f"{tag}.pm_init"] = digest(pm)
        mem, pm = dec(x[None, 2:3], pos[None, 2:3], ts[None, 2:3], mem)
        out[f"{tag}.pm_upd"] = digest(pm)
        out[f"{tag}.mem0"] = digest(mem[0][0])
        out[f"{tag}.mem11"] = digest(mem[0][11])
        out[f"{tag}.labels"] = mem[1][:, ::97].numpy()
        _, pm = dec(x[None], pos[None], ts[None], mem, render=True)
        out[f"{tag}.pm_render"] = digest(pm)
        print(tag, "done")
    np.savez_compressed(os.path.join(HERE, "full_model_digest.npz"), **out)


def chain_golden():
    """The benchmarked schedules, end to end through the reference ENGINE (engine/inference.py:370 inference_multi_ar, the
    call bench.py times): C3 = 20 views 512x384, mem_batches [2]+[1]*18, render all 20; C2 = 10 views 224x224, [2]+[1]*8,
    render all 10 (SURVEY.md 8d).  CPU fp32, SDPA branch, PyTorch RoPE fallback.  Digests only (strided samples + moments)."""
    out = {}
    for tag, (V, H, W, size) in {"c2": (10, 224, 224, 224), "c3": (20, 384, 512, 512)}.items():
        enc, dec = build_ref(dict(img_size=(size, size)),
                             dict(img_size=(size, size), feedback_type="single_mlp", memory_mode="kv",
                                  landscape_only=False), seed=0)
        imgs, ts = syn.synthetic_views(V, H, W, seed=2)
        views, tss = list(imgs.unbind(0)), list(ts.unbind(0))
        ids = [torch.tensor(i) for i in range(V)]
        raw = lambda pm: {"raw": pm}  # noqa: E731
        mem, pm0, pm = ref_engine.inference_multi_ar(enc, dec, views, ids, tss, [2] + [1] * (V - 2), max_bs=None,
                                                     post_process_function=raw, device="cpu", return_mem=True)
        raw_r = torch.stack([d["raw"] for d in pm])                       # [V,H,W,7] rendered
        raw_0 = torch.stack([d["raw"] for d in pm0])                      # first-pass predictions of the update calls
        post = ref_engine.postprocess(raw_r, ActivationType.NORM_EXP)
        out[f"{tag}.raw_render"] = digest(raw_r, 65536)
        out[f"{tag}.raw_first"] = digest(raw_0, 65536)
        out[f"{tag}.pts3d"] = digest(post["pts3d"], 32768)
        out[f"{tag}.pts3d_local"] = digest(post["pts3d_local"], 32768)
        out[f"{tag}.conf"] = digest(post["conf"], 32768)
        out[f"{tag}.raw_view_last"] = digest(raw_r[-1], 16384)            # the view that saw the longest chain
        out[f"{tag}.mem0"] = digest(mem[0][0], 16384)
        out[f"{tag}.mem11"] = digest(mem[0][11], 16384)
        out[f"{tag}.labels"] = mem[1][:, ::193].numpy()
        out[f"{tag}.tail"] = np.array(mem[2:], dtype=np.int64)
        print(tag, "done", flush=True)
    np.savez_compressed(os.path.join(HERE, "chain_digest.npz"), **out)


def engine_golden():
    """Engine schedulers (engine/inference.py) driven with the tiny reference model."""
    out = {}
    enc, dec = build_ref(TINY_ENC, TINY_DEC, seed=7)
    pp = lambda pm: ref_engine.postprocess(pm, ActivationType.NORM_EXP)  # noqa: E731
    # 6 views, two aspect ratios interleaved
    views = []
    for i in range(6):
        H, W = (32, 48) if i % 3 != 2 else (48, 32)
        im, ts = syn.synthetic_views(1, H, W, seed=100 + i)
        views.append((im[0], ts[0]))
    imgs = [v[0] for v in views]
    tss = [v[1] for v in views]
    img_ids = [torch.tensor(i) for i in range(6)]
    # offline: 4 keyframes in batches [2,1,1], one refinement iteration, render all 6
    mem, pm0, pm = ref_engine.inference_multi_ar(enc, dec, imgs, img_ids, tss, [2, 1, 1], max_bs=2,
                                                 post_process_function=pp, device="cpu", return_mem=True,
                                                 num_refinements_iterations=1)
    for i, d in enumerate(pm0):
        for k, v in d.items():
            out[f"multi_ar.pm0.{i}.{k}"] = v.numpy()
    for i, d in enumerate(pm):
        for k, v in d.items():
            out[f"multi_ar.pm.{i}.{k}"] = v.numpy()
    mem_arrays("multi_ar.mem", mem, out)
    # render-only call on a precomputed memory, subset of the views (engine/inference.py:370-527: precomputed_mem, to_render)
    _, pm_sel = ref_engine.inference_multi_ar(enc, dec, imgs, img_ids, tss, [2, 1, 1], max_bs=None, to_render=[5, 0, 2],
                                              precomputed_mem=mem, post_process_function=pp, device="cpu")
    for i, d in enumerate(pm_sel):
        for k, v in d.items():
            out[f"multi_ar.pm_sel.{i}.{k}"] = v.numpy()
    # video with one refinement pass (keyframe refresh + between-pass eviction), window of 3
    mem, pm0 = ref_engine.inference_video_multi_ar(enc, dec, imgs, tss, [2, 1, 1, 1, 1], max_bs=None,
                                                  post_process_function=pp, device="cpu", return_mem=True,
                                                  local_context_size=3, num_refinements_iterations=1)
    for i, d in enumerate(pm0):
        for k, v in d.items():
            out[f"video_ref.pm0.{i}.{k}"] = v.numpy()
    mem_arrays("video_ref.mem", mem, out)
    # video: rolling window of 2, keyframe iff id % 3 == 0 (engine/inference.py:236)
    mem, pm0 = ref_engine.inference_video_multi_ar(enc, dec, imgs, tss, [2, 1, 1, 1, 1], max_bs=None,
                                                  post_process_function=pp, device="cpu", return_mem=True,
                                                  local_context_size=2)
    for i, d in enumerate(pm0):
        for k, v in d.items():
            out[f"video.pm0.{i}.{k}"] = v.numpy()
    mem_arrays("video.mem", mem, out)
    # tensor path `inference` (engine/inference.py:595) with B=2 scenes of 4 views, chunked render
    im, ts = syn.synthetic_views(8, 32, 48, seed=200)
    pm0, pm = ref_engine.inference(enc, dec, im.view(2, 4, 3, 32, 48), ts.view(2, 4, 2), [2, 1, 1], max_bs=3)
    out["inference.pm0"], out["inference.pm"] = pm0.numpy(), pm.numpy()
    pm0b, pmb = ref_engine.inference(enc, dec, im.view(2, 4, 3, 32, 48), ts.view(2, 4, 2), [2, 1, 1], max_bs=None,
                                     to_render=[1, 3])
    out["inference.pm_sel"] = pmb.numpy()
    np.savez_compressed(os.path.join(HERE, "engine.npz"), **out)
    print("engine.npz", len(out), "arrays")


def keyframes_golden():
    """SLAM keyframe overlap scores (must3r/slam/model.py get_overlap_score, choose_keyframe_from_overlap) with the
    reference's scipy searchers (must3r/slam/nns.py), and its quadrant ids (must3r/slam/tools.py get_quadrant_id), on the
    seeded frames of tests/helpers.py -> tests/golden/keyframes.npz."""
    import importlib
    sys.path.insert(0, os.path.dirname(HERE))
    import helpers as h
    nns, model = importlib.import_module("must3r.slam.nns"), importlib.import_module("must3r.slam.model")
    tools = importlib.import_module("must3r.slam.tools")
    out = {}
    cam = torch.tensor(h.KEYFRAME_CAM)
    for method in h.KEYFRAME_METHODS:
        for mode in ("nn", "nn-norm"):
            tree = nns.get_searcher(method)
            for seed, shift in h.KEYFRAME_DB:
                fr = h.keyframe_frame(seed, shift=shift)
                tree.add_pts(fr["pts3d"][0, 0, ::2, ::2][fr["conf"][0, 0, ::2, ::2] > 1.5], cam_center=cam)
            for seed, shift in h.KEYFRAME_QUERIES:
                s = model.get_overlap_score(h.keyframe_frame(seed, shift=shift), tree, cam, mode=mode, kf_x_subsamp=2,
                                            min_conf_keyframe=1.5, percentile=70)
                out[f"{method}.{mode}.{seed}.score"] = np.float64(s)
                out[f"{method}.{mode}.{seed}.choice"] = np.bool_(model.choose_keyframe_from_overlap(s, 0.1, mode))
        s = model.get_overlap_score(h.keyframe_frame(60), nns.get_searcher(method), cam, mode="nn", kf_x_subsamp=2)
        out[f"{method}.empty.score"] = np.float64(s)
    fr = h.keyframe_frame(70)
    for mode in ("meanconf", "medianconf"):
        out[f"{mode}.score"] = np.float64(model.get_overlap_score(fr, None, None, mode=mode))
    rays = torch.randn(4000, 3, generator=torch.Generator().manual_seed(3))
    for div in (2, 4):
        out[f"quadrant{div}"] = np.asarray(tools.get_quadrant_id(rays.clone().numpy(), quadrant_divider=div)).astype(np.int8)
    np.savez_compressed(os.path.join(HERE, "keyframes.npz"), **out)
    print("keyframes.npz", len(out), "arrays")


def model_args_golden():
    """Constructor-string rewrites of load_model (must3r/model/__init__.py:53-108) -> tests/golden/model_args.json."""
    import json
    import must3r.model as ref_model
    encs = ["Dust3rEncoder(img_size=(512, 512), patch_embed='PatchEmbedDust3R')", "Dust3rEncoder(img_size=(224,224))",
            "Dust3rEncoder(img_size=(512,512),pos_embed='RoPE100')", "Dust3rEncoder(img_size=(512,512),pos_embed='RoPE100_224:512')",
            "MUSt3R(img_size=(512, 512), feedback_type='single_mlp', memory_mode=\"kv\", pos_embed='RoPE200_512:768', landscape_only=True)",
            "CausalMUSt3R(img_size=(224, 224), pos_embed='RoPE100', mem_dropout=0.1)"]
    decs = ["CausalMUSt3R(img_size=(512, 512), feedback_type='single_mlp', memory_mode=\"kv\", mem_dropout=0.1, "
            "dropout_mode='temporary', use_xformers_mask=True, use_mem_mask=True)",
            "MUSt3R(img_size=(512,512),landscape_only=True)", "MUSt3R(img_size=(512,512), landscape_only=False, head='Linear')"]
    out = {"set_image_size": [[e, sz, ref_model.set_image_size_in_args(e, sz, verbose=False)] for e in encs for sz in (224, 512, 768)],
           "convert": [[d, ref_model.convert_decoder_args(d)] for d in decs]}
    json.dump(out, open(os.path.join(HERE, "model_args.json"), "w"), indent=1)
    print("model_args.json", len(out["set_image_size"]) + len(out["convert"]), "cases")


if __name__ == "__main__":
    which = sys.argv[1:] or ["tiny", "engine", "full", "args"]
    if "args" in which:
        model_args_golden()
    if "tiny" in which:
        tiny_model_golden()
    if "engine" in which:
        engine_golden()
    if "full" in which:
        full_model_golden()
    if "chain" in which:
        chain_golden()
    if "keyframes" in which:
        keyframes_golden()
