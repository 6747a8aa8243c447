#!/usr/bin/env python
"""bench.py — views/sec of the MUSt3R multi-view inference hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3|c2|c4|c5] [--dtype bf16|fp16] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one whole job of a configuration of BASELINE.json (SURVEY.md §8d), on synthetic views and random-init
ViT-L encoder / ViT-B memory decoder:

  C2  MUSt3R_224, 10 views 224x224: encode, memory init with 2 views, 8 one-view updates, render 10, activation
  C3  MUSt3R_512, 20 views 512x384: encode, init 2, 18 one-view updates, render 20, activation   <- headline at N=1
  C4  ONE fixed scene of 100 views 512x384 (ceil-split over the N GPUs): sharded encoder, rounds of shard-local
      one-view updates whose new memory rows land in every GPU's memory (K|V GEMM epilogue -> NVLink peer stores),
      sharded render.  STRONG scaling: the headline at N>1, and an extra record at N=1.
  C5  online stream of 1000 frames 512x384, keyframe every 3rd frame, rolling window of 25 frames (1 GPU: the chain does
      not shard, SURVEY.md §8e), encoder look-ahead in batches.

Prints ONE JSON line (rank 0).  `value` = device-timed views/s with inputs resident in HBM; `e2e` = the same job through
the public engine API from pinned HOST images to HOST results (H2D / D2H inside the timed region); `parity` = rel-L2 of
the timed job's own outputs against the UNMODIFIED reference (oracle/_ref) run in fp32 on the same GPU, for fp16 and
bf16 operands; `roofline` = per-kernel-category achieved TFLOP/s vs the measured bf16 peak; `cpu_baseline` = the
unmodified reference's engine on this box's host cores on a bounded sample; `records` = the other configurations.
`--impl reference` times that CPU path alone.  `--dump-outputs DIR` writes what the last timed step returned (rank 0's
views) as DIR/<name>.npy; inputs and weights are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c2": dict(V=10, H=224, W=224, size=224, label="C2: MUSt3R_224 config, 10 synthetic views 224x224, init 2 + 8 one-view updates + render 10 + activation"),
    "c3": dict(V=20, H=384, W=512, size=512, label="C3: MUSt3R_512 config, 20 synthetic views 512x384, init 2 + 18 one-view updates + render 20 + activation"),
    "c4": dict(V=100, H=384, W=512, size=512, label="C4: ONE fixed scene of 100 synthetic views 512x384"),
    "c5": dict(V=1000, H=384, W=512, size=512, label="C5: online stream, 1000 synthetic frames 512x384, keyframe every 3rd, rolling window 25"),
}
# algorithmic GFLOP per view (multiply-add = 2), SURVEY.md §8a: encoder; decoder render a + b*M (M = memory views attended); update extra
FLOPS = {224: dict(enc=122.5e9, ren_a=41.1e9, ren_b=1.42e9, upd=12.9e9), 512: dict(enc=523.0e9, ren_a=177.3e9, ren_b=21.74e9, upd=50.7e9)}


def job_flops(size, n_enc, updates, renders):
    """updates / renders: lists of (n_views, memory views attended by each)."""
    f = FLOPS[size]
    return (f["enc"] * n_enc + sum(n * (f["ren_a"] + f["upd"] + f["ren_b"] * m) for n, m in updates)
            + sum(n * (f["ren_a"] + f["ren_b"] * m) for n, m in renders))


def chain_schedule(V):
    """[2] + [1]*(V-2): the init pair sees 1 peer view each, update k sees the k views already stored."""
    return [(2, 1)] + [(1, m) for m in range(2, V)], [(V, V)]


def split_counts(total, world):
    """ceil-split of `total` views over `world` ranks (the first ranks get the extra view)."""
    base, extra = divmod(total, world)
    return [base + (1 if r < extra else 0) for r in range(world)]


def sharded_schedule(counts):
    """Round s: every rank with a view s not yet stored updates it against the memory of the previous rounds."""
    upd, m_cur = [(2, 1)], 2
    for s in range(max(counts)):
        part = sum(1 for r, c in enumerate(counts) if s < c and not (r == 0 and s < 2))
        upd += [(1, m_cur)] * part
        m_cur += part
    tot = sum(counts)
    return upd, [(tot, tot)]


DUMP_BUDGET = 64 << 20


def dump_outputs(out, path, budget=DUMP_BUDGET):
    """Write the per-view result dicts a caller of the timed path receives, stacked over views, as <path>/<name>.npy in
    float32.  When the arrays exceed `budget` bytes in all, each keeps a fixed sample of its flattened elements (sorted
    indices drawn by numpy's default_rng(0), a share of the budget proportional to its size), so the files of two runs
    with the same arguments line up element for element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: torch.stack([d[k] for d in out]).float() for k in out[0]}
    total = sum(a.numel() for a in arrays.values()) * 4
    for k, a in arrays.items():
        if total > budget:
            n = a.numel()
            idx = np.unique(np.random.default_rng(0).integers(0, n, size=n * budget // total))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(path, f"{k}.npy"), a.cpu().numpy())
    return sorted(arrays)


def effective_cores():
    """Host threads for the CPU arm: bounded by sched affinity and the cgroup CPU quota (v2 and v1), then picked by a
    1-second calibration (fp32 2048^3 matmul at 4..64 threads) because oversubscribed boxes run slower with more threads."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda t: t.split()),
                        ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", lambda t: (t.strip(), open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().strip()))):
        try:
            q, per = parse(open(path).read())
            if q not in ("max", "-1"):
                n = min(n, max(1, int(float(q) / float(per))))
        except Exception:  # noqa: BLE001
            pass
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n}) or [1]
    a = torch.randn(2048, 2048)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.perf_counter()
        a @ a
        a @ a
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


class ClockSampler:
    def __init__(self, device_index):
        self.idx, self.rows, self._stop = device_index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        """NVML every 40 ms (a 5-step timed region is ~0.3 s); nvidia-smi every 200 ms if NVML is not importable."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.idx)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self._stop.is_set():
                r = int(get_reasons(h))
                flags = {n: ("Active" if r & b else "Not Active") for b, n in bits}
                self.rows.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx), flags["hw_slowdown"],
                                  flags["hw_thermal_slowdown"], flags["sw_thermal_slowdown"], flags["sw_power_cap"]])
                self._stop.wait(0.04)
            return
        except Exception:  # noqa: BLE001
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.t.join(timeout=10)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ reference (CPU arm, parity)
def reference_available():
    from baseline import ref_loader
    return ref_loader.available()


def build_reference(size, device, curope_shim):
    """The UNMODIFIED reference's classes (oracle/_ref, installed by oracle/install_reference.py) with the synthetic weights."""
    from baseline import ref_loader
    from must3r_b200 import synthetic as syn
    ref = ref_loader.load_reference(curope_shim=curope_shim)
    enc = ref.Dust3rEncoder(img_size=(size, size)).eval()
    dec = ref.MUSt3R(img_size=(size, size), feedback_type="single_mlp", memory_mode="kv", landscape_only=False).eval()
    enc.load_state_dict(syn.encoder_state_dict(0))
    dec.load_state_dict(syn.decoder_state_dict(0))
    return ref, enc.to(device), dec.to(device)


def cpu_reference_job(cfg, n_views, threads):
    """The reference's own engine on host cores (must3r/engine/inference.py:370 inference_multi_ar, SDPA branch, PyTorch RoPE
    fallback, fp32): the first `n_views` views of the configuration = encoder + 2-view init + (n-2) one-view updates +
    render of the n views + activation.  Falls back to the oracle port (kind "port") when oracle/_ref is absent."""
    from must3r_b200 import synthetic as syn
    torch.set_num_threads(threads)
    H, W, size = cfg["H"], cfg["W"], cfg["size"]
    imgs, ts = syn.synthetic_views(n_views, H, W, seed=2)
    views, tss, ids = list(imgs.unbind(0)), list(ts.unbind(0)), [torch.tensor(i) for i in range(n_views)]
    if reference_available():
        ref, enc, dec = build_reference(size, "cpu", curope_shim=False)
        pp = lambda pm: ref.engine.postprocess(pm, ref.model.ActivationType.NORM_EXP)  # noqa: E731

        def job():
            with torch.no_grad():
                return ref.engine.inference_multi_ar(enc, dec, views, ids, tss, [2] + [1] * (n_views - 2), max_bs=None,
                                                     post_process_function=pp, device="cpu")
        return job, "reference"
    from oracle import must3r_oracle as orc
    enc = orc.OracleEncoder(syn.encoder_state_dict(0), orc.EncoderConfig(img_size=(size, size)))
    dec = orc.OracleDecoder(syn.decoder_state_dict(0), orc.DecoderConfig(img_size=(size, size)))

    def job():
        x, pos = enc(imgs, ts)
        mem, _ = dec(x[None, :2], pos[None, :2], ts[None, :2], None)
        for i in range(2, n_views):
            mem, _ = dec(x[None, i:i + 1], pos[None, i:i + 1], ts[None, i:i + 1], mem)
        _, pm = dec(x[None], pos[None], ts[None], mem, render=True)
        return orc.postprocess(pm)
    return job, "port"


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cfg = CONFIGS["c3" if args.config in ("c4", "c5") else args.config]
    threads = effective_cores()
    n = args.cpu_views
    job, kind = cpu_reference_job(cfg, n, threads)
    for _ in range(args.warmup):
        job()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        job()
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    what = "unmodified reference (oracle/_ref, must3r.engine.inference_multi_ar, fp32, SDPA, RoPE fallback)" if kind == "reference" else "oracle port (oracle/_ref missing)"
    sample = f"{n} of the {cfg['V']} views per step ({cfg['H']}x{cfg['W']}: encoder + 2-view init + {n - 2} one-view update(s) + render {n} + activation), {what}"
    print(json.dumps({
        "impl": "reference", "metric": "views/sec at 512x384 (ViT-L enc / ViT-B dec)", "value": v, "unit": "views/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["label"], "views_per_step": n, "same_config": n == cfg["V"],
                   "cap": None if n == cfg["V"] else f"bounded sample: first {n} views of the schedule (a full job is minutes of CPU per step)"},
        "cpu_baseline": {"value": v, "unit": "views/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default=None, choices=list(CONFIGS), help="headline configuration (default: c3 at 1 GPU, c4 at N>1)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-views", type=int, default=3, help="views per step of the CPU reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-records", action="store_true", help="skip the extra configurations (records)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--stream-frames", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    ap.add_argument("--encoder-mode", default="precomputed", choices=["engine", "precomputed"],
                    help="precomputed (default): engine.encoder_multi_ar over all views first, then the decoder chain (features handed to "
                         "the engine); engine: encoder_precomputed_features=None, the engine encodes the missing views itself (up front, batched)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config is None:
        args.config = "c3" if world == 1 else "c4"
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    if world > 1 and args.config not in ("c4", "c5"):
        raise SystemExit("on more than one GPU: C4 (one scene, views sharded) or C5 (one stream, memory tokens sharded: context parallel)")

    import torch.distributed as dist
    from must3r_b200 import _lib, engine, synthetic as syn
    from must3r_b200.engine import sharded
    from must3r_b200.model import Dust3rEncoder, MUSt3R, set_precision, ActivationType

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    set_precision(dtype)
    lib = _lib.lib()
    pp = lambda pm: engine.postprocess(pm, ActivationType.NORM_EXP)  # noqa: E731
    models = {}

    def get_models(size):
        if size not in models:
            enc = Dust3rEncoder(img_size=(size, size))
            dec = MUSt3R(img_size=(size, size), feedback_type="single_mlp", memory_mode="kv", landscape_only=False)
            enc.load_state_dict(syn.encoder_state_dict(0))
            dec.load_state_dict(syn.decoder_state_dict(0))
            models[size] = (enc.to(dev).eval(), dec.to(dev).eval())
        return models[size]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup, sampler=None):
        """`warmup` untimed + `steps` timed calls of fn(), CUDA events on the launch stream, barrier + sync on both sides,
        max over ranks -> ms per step."""
        for _ in range(warmup):
            fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx = sampler if sampler is not None else _Null()
        with ctx:
            barrier()
            ev0.record()
            for _ in range(steps):
                fn()
            ev1.record()
            barrier()
        return max_over_ranks(ev0.elapsed_time(ev1) / steps)

    class _Null:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    # ---------------------------------------------------------------- jobs (public engine API)
    def make_chain_job(cfg):
        """C2 / C3 / C4 on one GPU: engine.encoder_multi_ar + engine.inference_multi_ar, schedule [2] + [1]*(V-2), render all."""
        V, H, W = cfg["V"], cfg["H"], cfg["W"]
        enc, dec = get_models(cfg["size"])
        imgs_host, ts = syn.synthetic_views(V, H, W, seed=2)
        state = {"dev": imgs_host.to(dev), "pinned": imgs_host.pin_memory(), "ts": ts}
        ids = [torch.tensor(i) for i in range(V)]

        def job(from_host=False, to_host=False, post=pp):
            imgs = state["pinned"].to(dev, non_blocking=True) if from_host else state["dev"]
            views, tss = list(imgs.unbind(0)), list(ts.unbind(0))          # true_shape stays on the host, as an image loader yields it
            feats = engine.encoder_multi_ar(enc, views, ts, device=dev, max_bs=50) if args.encoder_mode == "precomputed" else None
            _, pm = engine.inference_multi_ar(enc, dec, views, ids, tss, [2] + [1] * (V - 2), encoder_precomputed_features=feats,
                                              post_process_function=post, device=dev, preserve_gpu_mem=to_host)
            return pm
        upd, ren = chain_schedule(V)
        meta = {"views": V, "flops": job_flops(cfg["size"], V, upd, ren), "h2d": imgs_host.numel() * 4}
        return job, meta

    def make_sharded_job(cfg):
        """C4 on N GPUs: ONE scene, views ceil-split over the ranks (global order = rank-major)."""
        V, H, W = cfg["V"], cfg["H"], cfg["W"]
        enc, dec = get_models(cfg["size"])
        counts = split_counts(V, world)
        lo = sum(counts[:rank])
        imgs_all, ts_all = syn.synthetic_views(V, H, W, seed=2)
        imgs_host, ts = imgs_all[lo:lo + counts[rank]].contiguous(), ts_all[lo:lo + counts[rank]]
        state = {"dev": imgs_host.to(dev), "pinned": imgs_host.pin_memory()}

        def job(from_host=False, to_host=False, post=pp):
            imgs = state["pinned"].to(dev, non_blocking=True) if from_host else state["dev"]
            return sharded.inference_sharded(enc, dec, imgs, ts, post_process_function=post, device=dev, to_host=to_host,
                                             view_counts=counts)
        upd, ren = sharded_schedule(counts)
        meta = {"views": V, "flops": job_flops(cfg["size"], V, upd, ren), "h2d": imgs_host.numel() * 4, "counts": counts}
        return job, meta

    def make_stream_job(cfg, frames):
        """C5: engine.inference_video_multi_ar (keyframe iff id % 3 == 0, window 25), encoder look-ahead in batches of 50."""
        H, W = cfg["H"], cfg["W"]
        enc, dec = get_models(cfg["size"])
        if world > 1:
            # one stream on N GPUs: every rank runs the chain on the same frames, the memory TOKENS are sharded and every
            # cross-attention merges the ranks' partial states through peer memory (engine/context_parallel.py)
            from must3r_b200.engine.context_parallel import ContextParallelDecoder
            if "cp" not in models:
                models["cp"] = ContextParallelDecoder(dec)
            dec = models["cp"]
        imgs_host, ts = syn.synthetic_views(frames, H, W, seed=3)
        state = {"dev": imgs_host.to(dev)}
        del imgs_host

        def job(from_host=False, to_host=False, post=pp):
            views, tss = list(state["dev"].unbind(0)), list(ts.unbind(0))
            feats = engine.encoder_multi_ar(enc, views, ts, device=dev, max_bs=50) if args.encoder_mode == "precomputed" else None
            return engine.inference_video_multi_ar(enc, dec, views, tss, [2] + [1] * (frames - 2), encoder_precomputed_features=feats,
                                                   post_process_function=post, device=dev, local_context_size=25,
                                                   preserve_gpu_mem=to_host)
        # keyframes (every 3rd) stay, plus the <= 25 most recent frames: frame t attends ~ t/3 + min(t, 25)*2/3 views
        upd = [(2, 1)] + [(1, min(t, t // 3 + 1 + (min(t, 25) * 2) // 3)) for t in range(2, frames)]
        meta = {"views": frames, "flops": job_flops(cfg["size"], frames, upd, []), "h2d": 0}
        return job, meta

    # ---------------------------------------------------------------- parity of the timed job's outputs vs the reference
    def parity_record(tag, cfg, job):
        """rel-L2 of the job's rendered outputs (raw head, pts3d, conf) vs the unmodified reference run in fp32 on this GPU
        (TF32 off, its RoPE served by must3r_b200.compat.curope), for fp16 and bf16 operands.  Single-GPU chain configs."""
        if args.no_parity or not reference_available():
            return {"unavailable": "oracle/_ref missing" if not args.no_parity else "--no-parity"}
        V, H, W = cfg["V"], cfg["H"], cfg["W"]
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        ref, renc, rdec = build_reference(cfg["size"], dev, curope_shim=True)
        imgs, ts = syn.synthetic_views(V, H, W, seed=2)
        views, ids = list(imgs.to(dev).unbind(0)), [torch.tensor(i) for i in range(V)]
        raw = lambda pm: {"raw": pm}  # noqa: E731
        with torch.no_grad():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, rpm = ref.engine.inference_multi_ar(renc, rdec, views, ids, [t.to(dev) for t in ts.unbind(0)], [2] + [1] * (V - 2),
                                                   max_bs=None, post_process_function=raw, device=dev)
            torch.cuda.synchronize()
            t_ref = time.perf_counter() - t0
            r_raw = torch.stack([d["raw"] for d in rpm]).float()
            r_post = ref.engine.postprocess(r_raw, ref.model.ActivationType.NORM_EXP)
        del renc, rdec
        rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())  # noqa: E731
        out = {"against": "unmodified reference (oracle/_ref) fp32 on this GPU, TF32 off, same schedule through its own engine",
               "views": V, "reference_gpu_ms_per_job": round(t_ref * 1e3, 1)}
        for dt in (torch.float16, torch.bfloat16):
            set_precision(dt)
            pm = job(post=raw)
            o_raw = torch.stack([d["raw"] for d in pm]).float()
            o_post = engine.postprocess(o_raw, ActivationType.NORM_EXP)
            out["fp16" if dt == torch.float16 else "bf16"] = {
                "raw": rel(o_raw, r_raw), "pts3d": rel(o_post["pts3d"], r_post["pts3d"]),
                "pts3d_local": rel(o_post["pts3d_local"], r_post["pts3d_local"]), "conf": rel(o_post["conf"], r_post["conf"])}
        set_precision(dtype)
        torch.cuda.empty_cache()
        return out

    def sharded_parity(cfg, job, meta):
        """N>1: rank 0's rendered views vs the SAME schedule composed from single-process calls of the unmodified reference
        (fp32, rank 0's GPU): rounds of one-view updates against the memory of the previous rounds, tokens appended in rank
        order, then render (tests/test_sharded_cpu.py composes the oracle the same way)."""
        if args.no_parity or not reference_available():
            return {"unavailable": "oracle/_ref missing" if not args.no_parity else "--no-parity"}
        counts = meta["counts"]
        raw = lambda pm: {"raw": pm}  # noqa: E731
        res = {}
        pm = job(post=raw)                               # collective: every rank runs it
        if rank == 0:
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            ref, renc, rdec = build_reference(cfg["size"], dev, curope_shim=True)
            V, H, W = cfg["V"], cfg["H"], cfg["W"]
            imgs, ts = syn.synthetic_views(V, H, W, seed=2)
            imgs, ts = imgs.to(dev), ts.to(dev)
            with torch.no_grad():
                feats = [renc(imgs[i:i + 10], ts[i:i + 10]) for i in range(0, V, 10)]
                x, pos = torch.cat([f[0] for f in feats]), torch.cat([f[1] for f in feats])
                starts = [sum(counts[:r]) for r in range(world)]
                mem, _ = rdec(x[None, 0:2], pos[None, 0:2], ts[None, 0:2], None)
                for s in range(max(counts)):
                    parts = []
                    for r in range(world):
                        if s >= counts[r] or (r == 0 and s < 2):
                            continue
                        g = starts[r] + s
                        m2, _ = rdec(x[None, g:g + 1], pos[None, g:g + 1], ts[None, g:g + 1], mem)
                        Nm = mem[0][0].shape[1]
                        parts.append([v[:, Nm:] for v in m2[0]])
                    if parts:
                        vals = [torch.cat([mem[0][l]] + [p[l] for p in parts], 1) for l in range(len(mem[0]))]
                        n_new = len(parts)
                        N = x.shape[1]
                        lab = torch.cat([mem[1], (torch.arange(n_new, device=dev) + mem[2]).repeat_interleave(N)[None]], 1)
                        mem = (vals, lab, mem[2] + n_new, mem[3] + n_new, lab.shape[1])
                _, rpm = rdec(x[None, :counts[0]], pos[None, :counts[0]], ts[None, :counts[0]], mem, render=True)
            r_raw = rpm[0].float()
            o_raw = torch.stack([d["raw"] for d in pm]).float()
            rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())  # noqa: E731
            res = {"against": "sharded schedule composed from single-process calls of the unmodified reference (fp32, rank 0)",
                   "views_compared": int(counts[0]), args.dtype: {"raw": rel(o_raw, r_raw)}}
            del renc, rdec
            torch.cuda.empty_cache()
        return res

    # ---------------------------------------------------------------- headline
    cfg = CONFIGS[args.config]
    if args.config == "c5":
        job, meta = make_stream_job(cfg, args.stream_frames)
    elif world > 1:
        job, meta = make_sharded_job(cfg)
    else:
        job, meta = make_chain_job(cfg)
    launches0 = None
    clk = ClockSampler(local_rank)
    for _ in range(args.warmup):
        job()
    barrier()
    launches0 = lib.m3r_launch_count()
    last = {}

    def job_keep_output():
        last["out"] = job()
    ms = timed(job_keep_output if args.dump_outputs else job, args.steps, 0, sampler=clk)
    launches = (lib.m3r_launch_count() - launches0) // args.steps
    value = meta["views"] / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(last["out"], args.dump_outputs)
    last.clear()

    # ---- end to end: pinned host images -> host results (H2D / D2H inside the timed region)
    out = None

    def e2e_job():
        nonlocal out
        out = job(from_host=True, to_host=True)
    ms_e2e = timed(e2e_job, args.steps, 3)            # warm-up also brings the pinned staging pool to its steady state
    d2h = sum(v.numel() * v.element_size() for d in out for v in d.values())
    h2d_t = torch.tensor([float(meta["h2d"]), float(d2h)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(h2d_t)
    h2d, d2h = int(h2d_t[0].item()), int(h2d_t[1].item())

    # ---- profiled pass: per-category kernel time (CUDA events around every launch on the launch stream)
    roof, shares = None, None
    if rank == 0:
        lib.m3r_prof_enable(1)
    job()          # every rank runs it (the sharded job contains collectives); only rank 0 records
    torch.cuda.synchronize()
    if rank == 0:
        import ctypes as C
        buf = (C.c_double * 28)()
        lib.m3r_prof_read(buf)
        lib.m3r_prof_enable(0)
        cats = ["gemm BN>=256 (incl. CTA-pair)", "gemm BN 128..192", "gemm BN<=64 (incl. LN-emitting)", "attn_kernel<QT=2>", "attn_kernel<QT=1>+split-merge",
                "layernorm/normalize", "other"]
        prof = {c: {"ms": buf[i * 4], "launches": int(buf[i * 4 + 1]), "flops": buf[i * 4 + 2], "bytes": buf[i * 4 + 3]}
                for i, c in enumerate(cats)}
        tot_ms = sum(p["ms"] for p in prof.values()) or 1.0
        shares = {c: round(p["ms"] / tot_ms, 4) for c, p in prof.items()}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1590.0)) if peaks else 1590.0
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernels timed inside a long step)" if peaks else "fallback 1.59 PFLOP/s"
        tensor_cats = [c for c in cats if prof[c]["flops"] > 0]
        dom = max(tensor_cats, key=lambda c: prof[c]["ms"])
        ach = prof[dom]["flops"] / (prof[dom]["ms"] * 1e-3) / 1e12 if prof[dom]["ms"] > 0 else 0.0
        # dram__bytes_read + dram__bytes_write of ONE representative launch of the dominant category, taken from the committed
        # `ncu --set full` captures (bench.py cannot run ncu itself); the file names the launch shape and the summary it came from
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json"))).get(dom, {})
        except Exception:  # noqa: BLE001
            traffic = {}
        roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic.get("dram_bytes"), "traffic_of": traffic.get("launch"), "traffic_source": traffic.get("source"),
                "peak_source": peak_src,
                "note": "per-launch CUDA events serialise the side streams: the category times sum to more than the step; shares are indicative",
                "per_kernel": {c: {"ms": round(p["ms"], 3), "launches": p["launches"],
                                   "tflops": round(p["flops"] / (p["ms"] * 1e-3) / 1e12, 1) if p["ms"] > 0 and p["flops"] else None,
                                   "frac": round(p["flops"] / (p["ms"] * 1e-3) / 1e12 / peak, 4) if p["ms"] > 0 and p["flops"] else None}
                               for c, p in prof.items()}}
        roof["job_flops"] = meta["flops"]
        roof["job_tflops"] = meta["flops"] / (ms * 1e-3) / 1e12                  # aggregate over the N GPUs
        roof["job_tflops_per_gpu"] = roof["job_tflops"] / world
        roof["job_frac_of_peak"] = roof["job_tflops_per_gpu"] / peak

    # ---- parity of the timed job (both operand formats) and the other configurations
    if world > 1 and args.config == "c4":
        parity = sharded_parity(cfg, job, meta)
    elif args.config == "c5":
        parity = {"unavailable": "stream schedule: covered by the C3 / C2 records, tests/test_model_gpu.py::test_stream_schedule_* and tools/check_context_parallel.py"}
    else:
        parity = parity_record(args.config, cfg, job)
    records = {}
    if not args.no_records:
        def rec(tag, mk, steps, warm, with_parity):
            torch.cuda.empty_cache()
            j, m = mk()
            t = timed(j, steps, warm)
            r = {"workload": CONFIGS[tag]["label"], "views": m["views"], "ms_per_job": round(t, 3), "views_per_s": round(m["views"] / (t / 1e3), 2),
                 "job_tflops_per_gpu": round(m["flops"] / (t * 1e-3) / 1e12 / world, 1), "steps": steps, "warmup": warm, "dtype": args.dtype}
            if with_parity:
                r["parity"] = parity_record(tag, CONFIGS[tag], j)
            return r
        if world == 1:
            for tag in ("c2", "c3", "c4"):
                if tag == args.config:
                    continue
                records[{"c2": "c2_224_10views", "c3": "c3_512_20views", "c4": "c4_fixed100"}[tag]] = rec(
                    tag, lambda t=tag: make_chain_job(CONFIGS[t]), 3 if tag != "c4" else 2, 3 if tag != "c4" else 1, with_parity=(tag == "c2"))
            if args.config != "c5":
                fr = args.stream_frames
                r = rec("c5", lambda: make_stream_job(CONFIGS["c5"], fr), 1, 1, with_parity=False)
                r["frames"] = fr
                r["frames_per_s"] = r.pop("views_per_s")
                records["c5_stream"] = r
            if args.dtype == "bf16":                        # same kernels with fp16 operands (the 1e-3 parity mode)
                set_precision(torch.float16)
                t16 = timed(job, 3, 3)
                set_precision(dtype)
                records["headline_fp16_operands"] = {"ms_per_job": round(t16, 3), "views_per_s": round(meta["views"] / (t16 / 1e3), 2)}
        else:
            # strong scaling reference point measured in the same run: the same 100-view scene on rank 0 alone
            if rank == 0:
                j1, m1 = make_chain_job(cfg)
                for _ in range(1):
                    j1()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                j1()
                e1.record()
                torch.cuda.synchronize()
                t1 = e0.elapsed_time(e1)
                records["c4_fixed100_single_gpu_same_run"] = {"ms_per_job": round(t1, 3), "views_per_s": round(m1["views"] / (t1 / 1e3), 2),
                                                              "note": "reference chain [2]+[1]*98 on rank 0 alone (1 warm-up, 1 timed job)"}
            barrier()
            if args.config == "c4":
                # the stream configuration on the same GPUs: ONE stream, context-parallel cross-attention
                fr = args.stream_frames
                r = rec("c5", lambda: make_stream_job(CONFIGS["c5"], fr), 1, 1, with_parity=False)
                r["frames"], r["frames_per_s"] = fr, r.pop("views_per_s")
                r["parallelism"] = f"one stream replicated on {world} GPUs, memory tokens sharded round-robin, per-layer exchange of attention states over NVLink peer memory"
                r["job_tflops_per_gpu"] = None
                records["c5_stream_context_parallel"] = r
        records["c4_fixed100" if args.config == "c4" else "headline"] = {"ms_per_job": round(ms, 3), "views_per_s": round(value, 2), "n_gpus": world,
                                                                         "job_tflops_per_gpu": round(meta["flops"] / (ms * 1e-3) / 1e12 / world, 1)}

    # ---- CPU baseline on the host cores (rank 0, N=1 only), bounded sample.  Run in a fresh interpreter: this process has
    # imported the reference with the CUDA curope shim for the parity check, and the reference binds its RoPE at import time.
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ccfg_id = "c3" if args.config in ("c4", "c5") else args.config
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", ccfg_id, "--steps", "1",
                                "--warmup", "1", "--cpu-views", str(args.cpu_views)], capture_output=True, text=True, timeout=900,
                               env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            cpu = json.loads(line)["cpu_baseline"]
            cpu["sample"] += ", 1 run after 1 warm-up"
        except Exception as e:  # noqa: BLE001
            cpu = {"unavailable": f"reference arm failed: {type(e).__name__}: {e}"}

    if rank == 0:
        par = "single GPU" if world == 1 else (
            f"ONE stream on {world} GPUs: the chain is replicated, the memory tokens are sharded round-robin and every memory cross-attention "
            "merges the ranks' attention states exchanged through NVLink peer memory (context parallel)") if args.config == "c5" else (
            f"ONE scene of {meta['views']} views ceil-split over {world} GPUs {meta['counts']}: sharded encoder, rounds of shard-local one-view "
            "updates, new K|V rows stored into every GPU's memory by the GEMM epilogue over NVLink peer memory + one device-side "
            "flag barrier per round, sharded render")
        print(json.dumps({
            "metric": "views/sec at 512x384 (ViT-L enc / ViT-B dec)", "value": value, "unit": "views/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if args.config == "c4" else "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": cfg["label"] + (", random-init ViT-L enc / ViT-B dec" if True else ""), "config_id": args.config,
                       "global_views": meta["views"], "parallelism": par, "encoder_mode": args.encoder_mode,
                       "l2": "working set (1.7 GB of 16-bit weights + activations + memory tokens) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": meta["views"] / (ms_e2e / 1e3), "unit": "views/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches), "kernel_time_shares": shares, "roofline": roof, "parity": parity, "records": records,
            "cpu_baseline": cpu, "clocks": clk.summary()}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
