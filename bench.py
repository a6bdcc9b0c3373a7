#!/usr/bin/env python
"""bench.py -- frames/sec of the GeneFace++ render hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]                 # this repo's sm_100a kernels
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] # the reference's path on the host CPU cores
    python bench.py ... --dump-outputs DIR     # also write what the timed path returned in its last step as DIR/*.npy

One "step" = one pass of the hot path over one batch of synthetic input = rendering this rank's shard of a
512x512 head+torso clip (BASELINE config "May head+torso two-pass 512x512, 250 frames, 1xB200"; at N GPUs every
rank renders its own 250 frames -- config 4, 2000 frames over 8 GPUs -- and one NCCL all-gather of the RGB
follows: weak scaling).  Random-init May-shaped weights, synthetic poses/conditioning (no checkpoint or dataset
ships with the reference): "data": "synthetic".

Timed numbers:
  value      frames/s with inputs resident in HBM (poses, conditioning sequence, background), CUDA events,
             barrier + synchronize on both sides, max over ranks
  e2e        the same clip through the public clip API starting from pinned HOST buffers: H2D of poses +
             conditioning inside the timed region, D2H of the rendered uint8 frames
  roofline   dominant kernel (k_head, pass 1) timed live with CUDA events inside libgfpp on the launching
             stream: algorithmic bytes (SURVEY.md 8(d)) / duration vs the measured HBM peak
  cpu_baseline  the CPU oracle port timed on rank 0's host cores on a bounded sample of the same workload
"""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=250, help="frames per GPU per step")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--density-scale", type=float, default=8.0)
    ap.add_argument("--head-only", action="store_true")
    ap.add_argument("--frames-per-call", type=int, default=50)
    ap.add_argument("--cpu-frames", type=int, default=4, help="frames of the bounded CPU-baseline sample (~3.5 s each on the box)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-mode", action="store_true", help="skip measuring the other precision mode (fp16 <-> robust) beside the headline one")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip timing the reference's own CUDA kernels (oracle/_ref) beside ours")
    ap.add_argument("--no-sr-variants", action="store_true", help="skip the short measurement of the SR-checkpoint paths (SURVEY 8(f) rank 3)")
    ap.add_argument("--no-train-ops", action="store_true", help="skip timing the training-side native ops beside the reference's kernels (SURVEY 8(f) rank 4)")
    ap.add_argument("--precision", default=os.environ.get("GFPP_BENCH_PRECISION", DEFAULT_PRECISION), choices=["fp32", "fp16", "bf16x3", "bf16", "robust"],
                    help="arithmetic of the head MLP GEMMs (marching/gather/compositing are fp32 in every mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step as DIR/<name>.npy (at most ~56 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(path, clip, stats, H, W):
    """What the last timed step returned, so that two builds can be compared output for output on identical inputs:
    clip [F, H*W, 3] (fp32 frames at N = 1, the gathered uint8 clip at N > 1) and stats [F, 4] (B_total, n_survivors, S, P
    per frame).  A fixed, seeded sample of 2^21 clip values with their flat indices (24 MB), and up to 4 whole frames, at
    most 32 MB of them: at most ~56 MB in all."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    g = torch.Generator().manual_seed(0)
    flat = clip.reshape(-1)
    idx = torch.randint(0, flat.numel(), (min(flat.numel(), 1 << 21),), generator=g).sort().values
    k = min(4, clip.shape[0], (32 << 20) // (clip[0].numel() * 4))
    pick = torch.randperm(clip.shape[0], generator=g)[:k].sort().values
    arrays = {"clip_sample": flat[idx.to(flat.device)].float(), "clip_sample_index": idx.double(),
              "frames": clip[pick.to(clip.device)].float().reshape(k, H, W, 3), "frame_index": pick.double(), "stats": stats.double()}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured", d
    return 6650.0, "fallback", {}


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if "Active" in r[5 + k] and "Not" not in r[5 + k]:
                        reasons.add(nm)
            except Exception:
                pass
        if sm:
            busy = [s for s in sm if s > 0.5 * max(sm)] or sm
            out = {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except Exception:
            pass
        return out


_CPU_THREADS = None
DEFAULT_PRECISION = "fp16"                 # the headline mode of this bench
SMOKE_PRECISIONS = ("fp16", "robust")              # what __graft_entry__.smoke() renders beside the fp32 kernels


def metric_name(args):
    """ONE metric string for both arms (the driver pairs the two JSON lines by it)."""
    return f"frames/sec at {args.size}x{args.size} " + ("head" if args.head_only else "head+torso")


def cpu_reference_fps(args, n_frames, keep_images=False, rays=None):
    """The reference's path on the host cores: the reference's PyTorch-eager modules restated in oracle/render.py
    over the C restatement of its CUDA-only native ops (kind "port": the reference has no CPU implementation of
    those ops and its Python cannot travel to the GPU box).  All host threads."""
    import torch
    from genefaceplusplus_b200 import scene as scn
    from oracle import ops
    from oracle.render import OracleModel
    ops.build()
    cores = os.cpu_count() or 1
    sc = scn.Scene(H=args.size, W=args.size, T=max(n_frames, 8), torso=not args.head_only, density_scale=args.density_scale)
    orc = OracleModel(sc.state, sc.hparams)
    orc.density_scale = sc.density_scale
    # "all the host threads it can use": more threads than the op sizes can feed makes eager PyTorch slower, so the
    # thread count is calibrated on a small frame and the fastest setting is used (and reported)
    global _CPU_THREADS
    if _CPU_THREADS is None:
        cal = scn.Scene(H=96, W=96, T=8, torso=not args.head_only, density_scale=args.density_scale)
        co = OracleModel(cal.state, cal.hparams); co.density_scale = cal.density_scale
        fi = cal.frame_inputs(0)
        best = (1e30, cores)
        for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
            torch.set_num_threads(nt); ops.set_num_threads(nt)
            co.render(fi["rays_o"], fi["rays_d"], fi["cond"], fi["bg_coords"], fi["poses"], bg_color=fi["bg_color"], T_thresh=cal.T_thresh, **cal.hparams)
            t0 = time.time()
            co.render(fi["rays_o"], fi["rays_d"], fi["cond"], fi["bg_coords"], fi["poses"], bg_color=fi["bg_color"], T_thresh=cal.T_thresh, **cal.hparams)
            best = min(best, (time.time() - t0, nt))
        _CPU_THREADS = best[1]
    cores = _CPU_THREADS
    torch.set_num_threads(cores); ops.set_num_threads(cores)
    t0 = time.time()
    S = 0
    imgs, knife = [], []
    for t in range(n_frames):
        fi = sc.frame_inputs(t)
        # `rays`: ([F,N,3], [F,N,3]) CPU tensors to render instead of torch get_rays' -- the parity leg hands over the rays the GPU
        # path generated in-kernel, so that both sides see IDENTICAL rays (they differ from get_rays' by <= 2 ulp)
        ro, rd = (fi["rays_o"], fi["rays_d"]) if rays is None else (rays[0][t].view(1, -1, 3), rays[1][t].view(1, -1, 3))
        out = orc.render(ro, rd, fi["cond"], fi["bg_coords"], fi["poses"], bg_color=fi["bg_color"],
                         T_thresh=sc.T_thresh, **sc.hparams)
        S += out["stats"]["S"]
        if keep_images:
            imgs.append(out["rgb_map"].reshape(-1, 3).clone()); knife.append(out["knife"].reshape(-1).clone())
    dt = time.time() - t0
    if keep_images:
        return n_frames / dt, cores, dt, S, torch.stack(imgs), torch.stack(knife)
    return n_frames / dt, cores, dt, S


def measure_other_mode(args, sc, model, prec, poses_dev, pose6_dev, cond_dev, bg_color, bg_coords, rgb, hbm, S_per_frame, ref):
    """The other tensor-core precision mode on the SAME workload in the same run (N = 1): one timed step of the device-resident clip,
    its head-kernel roofline fraction, parity against the oracle frames of the cpu_baseline leg, and -- for both modes -- the max-abs
    error on the 'lively' well-conditioned scene (MLP gain 4, table amplitude ~ 1/resolution, 64x64) where plain fp16 does not hold 1e-3."""
    import ctypes
    import torch
    from genefaceplusplus_b200 import _capi, scene as scn
    from genefaceplusplus_b200.renderer import RADNeRF, RADNeRFTorso
    L = _capi.lib()
    H = W = args.size
    T = poses_dev.shape[0]
    cls = RADNeRF if args.head_only else RADNeRFTorso
    m = cls(sc.hparams); m.load_state_dict(sc.state, strict=True); m.density_scale = sc.density_scale; m.mlp_precision = prec
    m = m.to(poses_dev.device).eval()
    feat = m.cal_cond_feat_clip(cond_dev)[:T]
    kw = dict(cond_feat=feat, bg_color=bg_color, bg_coords=bg_coords, pose6=pose6_dev, T_thresh=sc.T_thresh, frames_per_call=args.frames_per_call, out=rgb)
    for _ in range(2):
        m.render_clip(poses_dev, sc.intrinsics, H, W, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); m.render_clip(poses_dev, sc.intrinsics, H, W, **kw); e1.record(); torch.cuda.synchronize()
    fps = T / (e0.elapsed_time(e1) / 1000.0)
    L.gfpp_profile_enable(1)
    Fc = min(args.frames_per_call, T)
    m.render_clip(poses_dev[:Fc], sc.intrinsics, H, W, **{**kw, "cond_feat": feat[:Fc], "pose6": None if pose6_dev is None else pose6_dev[:Fc], "out": rgb[:Fc]})
    buf = (ctypes.c_float * 4)(); _capi.check(L.gfpp_profile_read(buf), "profile_read")
    L.gfpp_profile_enable(0)
    head_t = buf[0] / 1000.0
    out = {"precision": prec, "value": fps, "unit": "frames/s", "steps": 1,
           "roofline_frac": Fc * (S_per_frame * 2048 + H * W * 20) / head_t / 1e9 / hbm, "head_launch_ms": buf[0]}
    if ref is not None:
        ref_img, ref_knife = ref
        Fp = ref_img.shape[0]
        mine = m.render_clip(poses_dev[:Fp], sc.intrinsics, H, W, **{**kw, "cond_feat": feat[:Fp], "pose6": None if pose6_dev is None else pose6_dev[:Fp], "out": None}).float().cpu()
        d = (mine - ref_img).abs().max(-1).values
        mse = ((mine.double() - ref_img.double()) ** 2).mean().item()
        out["parity"] = {"max_abs": d[~(ref_knife < 1e-3)].max().item(), "n_over_1e-3": int((d > 1e-3).sum()),
                         "psnr": 999.0 if mse == 0 else 10 * math.log10(1.0 / mse)}
        # lively scene, both modes, 64x64 against the oracle
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from helpers import lively_state
        from oracle.render import OracleModel
        ls = scn.Scene(H=64, W=64, T=4, torso=False, density_scale=1.0, table_decay=1.0, table_amp=1.0)
        st = lively_state(ls.state, 4.0)
        fi = ls.frame_inputs(0)
        orc = OracleModel(st, ls.hparams); orc.density_scale = ls.density_scale
        r = orc.render(fi["rays_o"], fi["rays_d"], fi["cond"], fi["bg_coords"], fi["poses"], bg_color=fi["bg_color"], T_thresh=ls.T_thresh, **ls.hparams)
        liv = {}
        for p in ("fp16", "robust"):
            lm = RADNeRF(ls.hparams); lm.load_state_dict(st, strict=True); lm.density_scale = ls.density_scale; lm.mlp_precision = p
            lm = lm.to(poses_dev.device).eval()
            o = lm.render(fi["rays_o"].cuda(), fi["rays_d"].cuda(), fi["cond"].cuda(), fi["bg_coords"].cuda(), fi["poses"].cuda(),
                          bg_color=fi["bg_color"].cuda(), T_thresh=ls.T_thresh, **ls.hparams)
            liv[p] = (o["rgb_map"].cpu().view(-1, 3) - r["rgb_map"].view(-1, 3)).abs().max().item()
        out["lively_scene_max_abs"] = liv
    return out


def workload_name(args):
    return (f"May {'head-NeRF' if args.head_only else 'head+torso two-pass'} {args.size}x{args.size}, {args.frames}-frame driving clip per GPU, "
            f"max_steps=16, T_thresh=0.01, density_scale={args.density_scale:g}")


def run_reference(args, out=sys.stdout):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fps_list = []
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_reference_fps(args, 1)
    cores = os.cpu_count() or 1
    t_total = 0.0
    for _ in range(args.steps):
        fps, cores, dt, _ = cpu_reference_fps(args, args.cpu_frames)
        fps_list.append(fps); t_total += dt
    v = args.cpu_frames * args.steps / t_total
    line = {"impl": "reference", "metric": metric_name(args), "value": v, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "sample": f"{args.cpu_frames} frame(s) of the clip per step"},
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(), "kind": "port",
                             "sample": f"{args.cpu_frames} frame(s) at {args.size}x{args.size} per step, {args.steps} steps",
                             "note": "oracle/render.py + oracle/native_ops.c (CPU restatement of the reference path; the reference's own Python "
                                     "has no CPU implementation of its native ops and does not travel to this box); `cores` = calibrated thread count"},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=out)


_T0 = time.time()


def _stage(msg):
    """Progress marks on stderr (GFPP_BENCH_VERBOSE=1): where a multi-rank run is when it is slow or stuck."""
    if os.environ.get("GFPP_BENCH_VERBOSE"):
        print(f"[bench r{os.environ.get('RANK', '0')} +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def _claim_stdout():
    """Keep stdout clean for the ONE JSON line: libraries (NCCL prints its version banner to stdout) are redirected to stderr."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    args = parse()
    out = _claim_stdout()
    try:
        return _main(args, out)
    finally:
        out.flush()


def _main(args, out):
    if args.impl == "reference":
        return run_reference(args, out)
    import torch
    import torch.distributed as dist
    from genefaceplusplus_b200 import _capi, scene as scn
    from genefaceplusplus_b200 import dist as gdist
    from genefaceplusplus_b200.renderer import RADNeRF, RADNeRFTorso

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the product path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _capi.lib()
    _capi.check(L.gfpp_check_device(), "gfpp_check_device")

    H = W = args.size
    T = args.frames
    sc = scn.Scene(H=H, W=W, T=T * world, torso=not args.head_only, density_scale=args.density_scale)
    model = (RADNeRF if args.head_only else RADNeRFTorso)(sc.hparams)
    model.load_state_dict(sc.state, strict=True)
    model.density_scale = sc.density_scale
    model.mlp_precision = args.precision
    model = model.to(dev).eval()
    s, e = gdist.frame_block(T * world, rank, world)
    poses_host = torch.stack([sc.pose(t) for t in range(s, e)]).pin_memory()
    cond_host = sc.cond.clone().pin_memory()            # full sequence on every rank (window halo)
    bg_color = sc.bg_color.to(dev)
    bg_coords = sc.bg_coords.to(dev)
    poses_dev = poses_host.to(dev)
    cond_dev = cond_host.to(dev)
    N = H * W
    rgb = torch.empty(T, N, 3, device=dev, dtype=torch.float32)
    u8 = torch.empty(T, N, 3, device=dev, dtype=torch.uint8)
    u8_host = torch.empty(T * world if rank == 0 else 1, N, 3, dtype=torch.uint8).pin_memory()
    launches = 0

    def step_device():
        nonlocal launches
        feat = model.cal_cond_feat_clip(cond_dev)[s:e]
        n0 = 0
        for a in range(0, T, args.frames_per_call):
            b = min(T, a + args.frames_per_call)
            # frames land in the clip buffer straight from the epilogue kernel: fp32 at N=1, the uint8 video frames at N>1
            # (what the all-gather moves)
            res = model.render_frames(feat[a:b], poses_c2w=poses_dev[a:b], intrinsics=sc.intrinsics, H=H, W=W,
                                      pose6=pose6_dev[a:b] if not args.head_only else None, bg_coords=bg_coords, bg_color=bg_color,
                                      dt_gamma=sc.hparams["dt_gamma"], max_steps=sc.hparams["max_steps"], T_thresh=sc.T_thresh,
                                      want_torso_maps=False, want_stats=True, want_aux=False,
                                      **({"u8_out": u8[a:b]} if world > 1 else {"rgb_out": rgb[a:b]}))
            stats_acc.append(res["stats"])
            n0 += model.last_launch_count
        launches += n0
        if world > 1:
            return gdist.gather_frames(u8, T * world)      # ONE all-gather of the uint8 clip (north_star)
        return rgb

    def step_e2e():
        """The call a user makes, from HOST buffers: H2D of this rank's poses + the conditioning sequence, euler/translation
        conversion of the poses, conditioning nets, render (uint8 frames written by the epilogue kernel), at N>1 the all-gather of
        the uint8 clip, and the D2H of the finished clip (whole clip on rank 0)."""
        p = poses_host.to(dev, non_blocking=True)
        c = cond_host.to(dev, non_blocking=True)
        p6 = scn.convert_poses(poses_host).to(dev, non_blocking=True) if not args.head_only else None
        cf = model.cal_cond_feat_clip(c)[s:e]
        out = model.render_clip(p, sc.intrinsics, H, W, cond_feat=cf, bg_color=bg_color, bg_coords=bg_coords, pose6=p6,
                                T_thresh=sc.T_thresh, frames_per_call=args.frames_per_call, out=u8, as_uint8=True)
        if world > 1:
            out = gdist.gather_frames(out, T * world)
        if rank == 0:
            u8_host.copy_(out, non_blocking=True)

    pose6_dev = scn.convert_poses(poses_host).to(dev) if not args.head_only else None
    stats_acc = []

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing ----------------
    _stage("setup done, warm-up")
    for _ in range(max(args.warmup, 3)):
        step_device()
    sync_all()
    _stage("warm-up done, timing")
    stats_acc.clear(); launches = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record()
    for _ in range(args.steps):
        last = step_device()
    ev1.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else {}
    if rank == 0 and args.dump_outputs:
        # before the legs below reuse the clip buffer
        dump_outputs(args.dump_outputs, last, torch.cat(stats_acc, 0)[-T:], H, W)
    ms = ev0.elapsed_time(ev1)
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = tms.item()
    timed_launches = launches
    st = torch.cat(stats_acc, 0).cpu()   # [steps*T, 4]: B_total, n_survivors, S, P
    S_per_frame = st[:, 2].float().mean().item()
    P_per_frame = st[:, 3].float().mean().item()
    fps = world * T * args.steps / (ms / 1000.0)

    _stage("device-resident timing done")
    # ---------------- dominant-kernel roofline (live, CUDA events inside libgfpp) ----------------
    L.gfpp_profile_enable(1)
    head_ms, pass2_ms, epi_ms, pre_ms = [], [], [], []
    feat = model.cal_cond_feat_clip(cond_dev)[s:e]
    Fc = min(args.frames_per_call, T)
    for it in range(5):
        model.render_frames(feat[:Fc], poses_c2w=poses_dev[:Fc], intrinsics=sc.intrinsics, H=H, W=W,
                            pose6=pose6_dev[:Fc] if not args.head_only else None, bg_coords=bg_coords, bg_color=bg_color,
                            dt_gamma=sc.hparams["dt_gamma"], max_steps=sc.hparams["max_steps"], T_thresh=sc.T_thresh, want_torso_maps=False)
        buf = (ctypes.c_float * 4)()
        _capi.check(L.gfpp_profile_read(buf), "profile_read")
        if it >= 2:
            head_ms.append(buf[0]); pass2_ms.append(buf[1]); epi_ms.append(buf[2]); pre_ms.append(buf[3])
    L.gfpp_profile_enable(0)
    hbm, peak_kind, pk = peaks()
    head_t = statistics.mean(head_ms) / 1000.0
    # SURVEY.md 8(d): 2 grids x 16 levels x 8 corners x 8 B per valid sample; per ray 12 B colour + 4 B alpha + 4 B depth out
    # (+24 B when rays are supplied: here they are generated in-kernel); + the packed weights once
    alg_bytes = Fc * (S_per_frame * 2048 + N * (12 + 4 + 4)) + 0.36e6
    alg_flops = Fc * S_per_frame * 178944
    achieved = alg_bytes / head_t / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if args.precision in tj:
            traffic = tj[args.precision]["dram_bytes_per_frame"] * Fc
            traffic_src = "static: " + tj[args.precision]["source"] + " (not measured in this run; scaled to this launch size)"
    # what physically moves: the fp16 / int16 'oct' layouts hold the 8 corners of a cell in ONE 32-byte sector per (sample, level),
    # the fp32 'quad' layout in two; everything is L2-resident, so the binding resources are L1/L2 sector rate and the tensor pipe
    sectors_per_sample = 2 * 16 * (1 if args.precision in ("fp16", "robust") else 2)
    sm_hz = 1e6 * (clocks.get("sm_mhz") or 1965.0) if rank == 0 else 1.965e9
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    sector_rate = Fc * S_per_frame * sectors_per_sample / head_t          # sectors / s
    bf16_peak = (pk.get("bf16_tflops_sustained") or 1460.6)
    kname = {"fp32": "k_head (pass 1)", "bf16": "k_head_tc (pass 1)", "bf16x3": "k_head_tc (pass 1)"}.get(args.precision, "k_head_v2 (pass 1)")
    if os.environ.get("GFPP_HEAD_V1"):
        kname = "k_head_tc (pass 1)"
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": hbm, "peak_source": peak_kind, "unit": "GB/s",
                "frac": achieved / hbm, "traffic": traffic, "traffic_source": traffic_src, "launch_ms": head_t * 1000.0, "frames_per_launch": Fc,
                "share_of_step": head_t / (head_t + (statistics.mean(pass2_ms) + statistics.mean(epi_ms) + statistics.mean(pre_ms)) / 1000),
                "ray_setup_ms": statistics.mean(pre_ms),
                "fp32_tflops": alg_flops / head_t / 1e12, "pass2_ms": statistics.mean(pass2_ms), "epilogue_ms": statistics.mean(epi_ms),
                "alg_bytes_per_frame": alg_bytes / Fc, "alg_flops_per_frame": alg_flops / Fc,
                "gathered_bytes_per_frame": S_per_frame * sectors_per_sample * 32,
                "l2_sector_frac": sector_rate / (1.0 * n_sm * sm_hz),
                "l2_sector_note": "scattered 32-byte sectors per second / (1.0 sector per clock per SM: the measured ceiling, profiles/microbench_gather_r01.txt)",
                "tensor_frac": alg_flops / head_t / 1e12 / bf16_peak,
                "tensor_note": "algorithmic MLP flops per second / measured sustained dense bf16 peak (MEASURED_PEAKS.json)"}

    # ---------------- end to end (host buffers in, uint8 frames out) ----------------
    _stage("roofline leg done, end-to-end")
    for _ in range(2):
        step_e2e()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    sync_all()
    ems = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_fps = world * T * args.steps / (ems.item() / 1000.0)
    _stage("end-to-end done")
    h2d = poses_host.numel() * 4 + cond_host.numel() * 4 + (0 if args.head_only else T * 6 * 4)
    d2h = u8_host.numel()

    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        Fp = args.cpu_frames
        kro, krd = model.generate_rays(poses_dev[:Fp], sc.intrinsics, H, W)      # the rays the clip path generates in-kernel
        v, cores, dt, _, ref_img, ref_knife = cpu_reference_fps(args, args.cpu_frames, keep_images=True, rays=(kro.cpu(), krd.cpu()))
        cpu = {"value": v, "unit": "frames/s", "cores": cores, "host_cores": os.cpu_count(), "kind": "port",
               "sample": f"{args.cpu_frames} frame(s) of the same clip at {H}x{W} ({dt:.1f} s)",
               "note": "oracle/render.py + oracle/native_ops.c on the host cores (the reference's Python has no CPU path for its native ops "
                       "and does not travel to this box); `cores` = calibrated thread count, `host_cores` = os.cpu_count()"}
        # parity of the BENCHMARKED configuration: the same frames through the timed path (clip API, in-kernel rays, timed
        # precision) against the fp32 CPU oracle's frames just rendered for the baseline (SURVEY 8(d): max-abs 1e-3 / PSNR 50 dB)
        mine = model.render_clip(poses_dev[:Fp], sc.intrinsics, H, W, cond_feat=model.cal_cond_feat_clip(cond_dev)[s:s + Fp],
                                 bg_color=bg_color, bg_coords=bg_coords, pose6=pose6_dev[:Fp] if not args.head_only else None,
                                 T_thresh=sc.T_thresh, frames_per_call=args.frames_per_call).float().cpu()
        d = (mine - ref_img).abs().max(-1).values                       # [F,N]
        knife = ref_knife < 1e-3                                         # rays whose termination an fp32 reordering may flip
        mse = ((mine.double() - ref_img.double()) ** 2).mean().item()
        parity = {"vs": "fp32 CPU oracle (oracle/render.py) on IDENTICAL rays (the in-kernel generated ones, exported through gfpp_debug_generate_rays: "
                        "<= 2 ulp from torch get_rays) and identical conditioning",
                  "precision": args.precision, "frames": Fp, "size": H,
                  "max_abs": d[~knife].max().item(), "max_abs_all": d.max().item(), "n_knife": int(knife.sum()),
                  "n_over_1e-3": int((d > 1e-3).sum()), "n_pixels": d.numel(),
                  "psnr": 999.0 if mse == 0 else 10 * math.log10(1.0 / mse), "tolerance": {"max_abs": 1e-3, "psnr": 50.0}}
        parity["ok"] = bool(parity["max_abs"] <= 1e-3 and parity["psnr"] >= 50.0)
    gpu_ref = None
    if rank == 0 and not args.no_gpu_reference:
        # SURVEY 8(d)(ii): the reference's own CUDA kernels (oracle/_ref, built unmodified) under its host loop, same box, same run
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import ref_gpu_baseline
            if ref_gpu_baseline.available():
                precs = ("fp32", args.precision) if args.precision != "fp32" else ("fp32",)
                gpu_ref = ref_gpu_baseline.measure(H, 8, args.density_scale, precisions=precs, torso=not args.head_only)
            else:
                gpu_ref = {"unavailable": "oracle/_ref/*.so not present (they are built where /root/reference exists and travel with the repo)"}
        except Exception as ex:   # a baseline measurement must never take the bench down
            gpu_ref = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    other = None
    if rank == 0 and world == 1 and not args.no_other_mode and args.precision in ("fp16", "robust"):
        other = measure_other_mode(args, sc, model, "robust" if args.precision == "fp16" else "fp16", poses_dev, pose6_dev, cond_dev, bg_color, bg_coords,
                                   rgb, hbm, S_per_frame, (ref_img, ref_knife) if parity is not None else None)
    sr = None
    if rank == 0 and world == 1 and not args.no_sr_variants:
        # SURVEY 8(f) rank 3, measured in the same run: the SR checkpoints' clip paths (NeRF at 256x256 + torso-SR field + 256->512 SR
        # head on tcgen05), every stage in libgfpp, beside the SR head as host-side PyTorch / cuDNN (tools/sr_bench.py)
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import sr_bench
            sr = {"config": "256x256 NeRF (fp16 tcgen05) -> 512x512, 32-frame clips, resident inputs, CUDA events, median of 3", "results": sr_bench.measure(32, 3)}
        except Exception as ex:   # an extra measurement must never take the bench down
            sr = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    train = None
    if rank == 0 and world == 1 and not args.no_train_ops:
        # SURVEY 8(f) rank 4, measured in the same run: libgfpp's training-side ops beside the reference's own training kernels
        # (oracle/_ref) on the same inputs (tools/train_bench.py).  Last measurement of the run: nothing depends on it.
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import train_bench
            train = train_bench.measure(256, 5)
        except Exception as ex:   # an extra measurement must never take the bench down
            train = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    if rank == 0:
        line = {"metric": metric_name(args), "value": fps,
                "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp32": "f32", "fp16": "f16 operands, f32 accumulate (tcgen05)", "bf16x3": "bf16 hi/lo split x3, f32 accumulate (tcgen05)", "bf16": "bf16 operands, f32 accumulate (tcgen05)",
                          "robust": "f16 operands, f32 accumulate (tcgen05); hi/lo split x3 on the ambient net, 16-bit fixed-point position table"}[args.precision],
                "data": "synthetic",
                "config": {"workload": workload_name(args), "mlp_precision": args.precision, "frames_per_gpu_per_step": T, "frames_per_call": args.frames_per_call,
                           "S_valid_samples_per_frame": S_per_frame, "P_torso_pixels_per_frame": P_per_frame, "B_total": int(st[0, 0]),
                           "parallelism": f"frame-sharded x{world}, one NCCL all-gather of the uint8 clip at the end" if world > 1 else "single GPU",
                           "l2": "per-step working set (786 MB fp32 frames out + 1.8 GB workspace) >> 126 MB L2; grid tables (14.4 MB) are L2-resident by design"},
                "clocks": clocks, "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                          "note": "pinned host poses+conditioning in (H2D, pose conversion and conditioning nets inside the timed "
                                                  "region), uint8 [T,H,W,3] frames written by the epilogue kernel" +
                                                  (", all-gather of the uint8 clip, D2H of the whole clip on rank 0" if world > 1 else ", D2H of the clip")},
                "gpu_launches": timed_launches, "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "gpu_reference": gpu_ref,
                "other_mode": other, "sr_variants": sr, "train_ops": train}
        print(json.dumps(line), file=out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
