"""Run under torchrun on N GPUs: the sharded schedule (engine.sharded.inference_sharded: fused GEMM -> peer stores with the
device-side flag barrier, or NCCL all-gather with M3R_FUSED_GATHER=0) must
  (1) reproduce, bit for bit, the same schedule composed from single-process CUDA decoder calls, with identical memory on
      all ranks - also on a second call that reuses the cached peer arena, and with a ragged split of the views;
  (2) match the schedule composed from single-process calls of the UNMODIFIED reference (oracle/_ref, fp32 on this GPU)
      at 512x384 within the fp16-operand tolerance (SURVEY.md 8e oracle).
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/check_sharded.py"""
import os, sys
import torch
import torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from must3r_b200 import synthetic as syn  # noqa: E402
from must3r_b200.engine import sharded  # noqa: E402
from must3r_b200.model import Dust3rEncoder, MUSt3R, set_precision  # noqa: E402

rank, world, lrank = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lrank)
dev = torch.device("cuda", lrank)
dist.init_process_group("nccl", device_id=dev)
ok_all = True


def composed(dec_call, upd_call, feats, counts):
    """The sharded schedule from single-process calls: init on rank 0's first two views, rounds of one-view updates against the
    memory of the previous rounds (tokens appended in rank order)."""
    x0, p0, t0 = feats[0]
    m, _ = dec_call(x0[None, :2], p0[None, :2], t0[None, :2], None)
    m = list(m)
    for s in range(max(counts)):
        parts = []
        for r in range(world):
            if (r == 0 and s < 2) or s >= counts[r]:
                continue
            x, pos, t = feats[r]
            parts.append(upd_call(x[None, s:s + 1], pos[None, s:s + 1], t[None, s:s + 1], tuple(m)))
        if not parts:
            continue
        N = parts[0][0].shape[1]
        m[0] = [torch.cat([m[0][l]] + [p[l] for p in parts], 1) for l in range(len(m[0]))]
        lab = torch.arange(m[2], m[2] + len(parts), device=dev).repeat_interleave(N)[None]
        m[1] = torch.cat([m[1], lab], 1); m[2] = m[3] = m[2] + len(parts); m[4] = m[1].shape[1]
    return tuple(m)


def run_case(tag, size, H, W, depth_e, depth_d, counts, dtype, calls=1, vs_reference=False):
    global ok_all
    set_precision(dtype)
    enc = Dust3rEncoder(img_size=(size, size), depth=depth_e)
    dec = MUSt3R(img_size=(size, size), depth=depth_d, feedback_type="single_mlp", memory_mode="kv", landscape_only=False)
    esd, dsd = syn.encoder_state_dict(3, depth=depth_e), syn.decoder_state_dict(3, depth=depth_d)
    enc.load_state_dict(esd); dec.load_state_dict(dsd)
    enc, dec = enc.to(dev).eval(), dec.to(dev).eval()
    views = [syn.synthetic_views(max(counts), H, W, seed=400 + r) for r in range(world)]
    views = [(v[0][:counts[r]].contiguous(), v[1][:counts[r]].contiguous()) for r, v in enumerate(views)]
    imgs, ts = views[rank][0].to(dev), views[rank][1].to(dev)
    for c in range(calls):
        mem, outs = sharded.inference_sharded(enc, dec, imgs, ts, device=dev, return_mem=(c == calls - 1), view_counts=counts) \
            if c == calls - 1 else (None, sharded.inference_sharded(enc, dec, imgs, ts, device=dev, view_counts=counts))
        outs = torch.stack(outs)
        if c == 0:
            first = outs.clone()
        else:
            assert torch.equal(first, outs), "second call on the cached arena differs"
    feats = []
    for r in range(world):
        x, pos = enc(views[r][0].to(dev), views[r][1].to(dev)); feats.append((x, pos, views[r][1].to(dev)))
    m = composed(lambda *a: dec(*a), lambda *a: dec.update_tokens(*a)[0], feats, counts)
    x, pos, t = feats[rank]
    _, pm = dec(x[None], pos[None], t[None], m, render=True)
    err = float((outs - pm[0]).norm() / pm[0].norm())
    mem_equal = all(torch.equal(mem[0][l], m[0][l]) for l in range(len(m[0]))) and torch.equal(mem[1], m[1])
    chk = torch.stack([mm.float().sum() for mm in mem[0]])
    allc = [torch.empty_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    same = all(torch.equal(allc[0], c) for c in allc)
    msg = f"[{tag}] rank {rank}/{world} counts {counts}: render rel err vs composed CUDA schedule {err:.3e}; memory == composed: {mem_equal}; identical on all ranks: {same}; Nmem {mem[1].shape[1]}"
    ok = err < 1e-5 and mem_equal and same
    if vs_reference:
        from baseline import ref_loader
        if ref_loader.available():
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            ref = ref_loader.load_reference(curope_shim=True)
            renc = ref.Dust3rEncoder(img_size=(size, size), depth=depth_e).eval()
            rdec = ref.MUSt3R(img_size=(size, size), depth=depth_d, feedback_type="single_mlp", memory_mode="kv", landscape_only=False).eval()
            renc.load_state_dict(esd); rdec.load_state_dict(dsd)
            renc, rdec = renc.to(dev), rdec.to(dev)
            with torch.no_grad():
                rfeats = []
                for r in range(world):
                    rx, rpos = renc(views[r][0].to(dev), views[r][1].to(dev)); rfeats.append((rx, rpos, views[r][1].to(dev)))

                def upd(x_, p_, t_, m_):
                    Nm = m_[0][0].shape[1]
                    m2, _ = rdec(x_, p_, t_, m_)
                    return [v[:, Nm:] for v in m2[0]]
                rm = composed(lambda *a: rdec(*a), upd, rfeats, counts)
                rx, rpos, rt = rfeats[rank]
                _, rpm = rdec(rx[None], rpos[None], rt[None], rm, render=True)
            e_ref = float((outs.double() - rpm[0].double()).norm() / rpm[0].double().norm())
            e_mem = float((mem[0][-1].double() - rm[0][-1].double()).norm() / rm[0][-1].double().norm())
            gate = 1.2e-3 if dtype == torch.float16 else 1.1e-2
            msg += f"; vs composed UNMODIFIED reference (fp32): render {e_ref:.2e}, last-level memory {e_mem:.2e} (gate {gate:.1e})"
            ok = ok and e_ref < gate and e_mem < 1.3 * gate
        else:
            msg += "; oracle/_ref missing: reference composition skipped"
    print(msg, flush=True)
    ok_all = ok_all and ok


even = [3] * world
ragged = [3] + [2] * (world - 1)
run_case("224 small model, even split, 3 calls (2 on the cached arena)", 224, 224, 224, 6, 4, even, torch.bfloat16, calls=3)
run_case("224 small model, ragged split", 224, 224, 224, 6, 4, ragged, torch.bfloat16)
run_case("512x384 full model, ragged split, vs reference", 512, 384, 512, 24, 12, ragged, torch.float16, vs_reference=True)
dist.barrier(); dist.destroy_process_group()
sys.exit(0 if ok_all else 1)
