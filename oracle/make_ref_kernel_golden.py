"""Writes tests/golden/ref_kernels.npz: what the reference's OWN CUDA kernels (oracle/_ref, compiled unmodified by
oracle/build_ref.py) return on the inputs of tests/test_gpu_ref_pin.py and of the reference pin in tests/test_gpu_train_ops.py.

Runs only on a GPU where oracle/_ref has been built:

    python -m oracle.make_ref_kernel_golden [--out tests/golden/ref_kernels.npz]

The tests rebuild the same inputs (the builders below), check them against the SHA-256 digests stored in `meta`, and hold the
C checker (and libgfpp) to the stored outputs, so they need neither the reference nor its kernels.  Outputs too large to store
whole are kept as a fixed sample: the indices of the sampled rows / entries are stored beside them.
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "ref_kernels.npz")


def digest(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def sample(n, k, seed):
    """k distinct sorted indices out of range(n) (all of them when k >= n)."""
    if k >= n:
        return np.arange(n, dtype=np.int32)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False)).astype(np.int32)


# ------------------------------------------------------------------------------------------------ inputs (shared with the tests)
def march_inputs():
    from genefaceplusplus_b200 import scene as scn
    sc = scn.Scene(H=96, W=96, T=4, torso=False)
    fi = sc.frame_inputs(1)
    return sc, fi["rays_o"].view(-1, 3).contiguous(), fi["rays_d"].view(-1, 3).contiguous()


def composite_inputs():
    g = torch.Generator().manual_seed(5)
    N, n_alive, n_step = 400, 256, 4
    alive = torch.randperm(N, generator=g)[:n_alive].int().contiguous()
    M = n_alive * n_step
    sig = torch.rand(M, generator=g) * 30; rgb = torch.rand(M, 3, generator=g)
    deltas = torch.stack([torch.full((M,), 0.027), torch.rand(M, generator=g) + 3], -1).contiguous()
    ws = torch.rand(N, generator=g) * 0.8; dp = torch.rand(N, generator=g); img = torch.rand(N, 3, generator=g); t = torch.rand(N, generator=g)
    return n_alive, n_step, alive, t, ws, dp, img, sig, rgb, deltas


def grid_inputs(D):
    from genefaceplusplus_b200.config import GridLayout
    lay = GridLayout(D)
    g = torch.Generator().manual_seed(D)
    emb = torch.rand(lay.n_entries, 2, generator=g) - 0.5
    x = torch.rand(8192, D, generator=g)
    return lay, emb, x, torch.from_numpy(lay.offsets.copy())


def sh_freq_inputs():
    g = torch.Generator().manual_seed(0)
    d = torch.nn.functional.normalize(torch.randn(4096, 3, generator=g), dim=-1)
    x = (torch.rand(2048, 2, generator=g) * 2 - 1) * 0.8
    return d, x


def train_rays(oracle_ops, H=64):
    from genefaceplusplus_b200 import scene as scn
    sc = scn.Scene(H=H, W=H, T=2, torso=False)
    fi = sc.frame_inputs(1)
    ro, rd = fi["rays_o"].view(-1, 3).contiguous(), fi["rays_d"].view(-1, 3).contiguous()
    nears, fars = oracle_ops.near_far_from_aabb(ro, rd, sc.state["aabb_infer"], 0.05)
    return sc, ro, rd, nears, fars


def segments(N=3000, seed=0, max_len=40):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, max_len, (N,), generator=g, dtype=torch.int32)
    lens[::7] = 0
    lens[3] = 70
    offs = torch.cumsum(lens.long(), 0) - lens.long()
    perm = torch.randperm(N, generator=g).int()
    rays = torch.stack([perm, offs.int(), lens], 1).contiguous()
    M = int(lens.sum())
    sig = torch.rand(M, generator=g) * 6
    rgb = torch.rand(M, 3, generator=g)
    amb = torch.rand(M, generator=g)
    dt = torch.rand(M, generator=g) * 0.05 + 0.01
    deltas = torch.stack([dt, torch.rand(M, generator=g) * 3 + 2], 1).contiguous()
    return rays, M, sig, rgb, amb, deltas


def train_grid_inputs():
    """Composite-backward upstream gradients first, then the grid inputs, from ONE generator (the order the pin draws them)."""
    from genefaceplusplus_b200.config import GridLayout
    Ns = segments()[0].shape[0]
    g = torch.Generator().manual_seed(9)
    gws, gas, gim = torch.randn(Ns, generator=g), torch.randn(Ns, generator=g), torch.randn(Ns, 3, generator=g)
    lay = GridLayout(3, log2_hashmap_size=16, desired_resolution=2048, gridtype="tiled")
    offsets = torch.from_numpy(np.asarray(lay.offsets, dtype=np.int32))
    table = torch.rand(int(offsets[-1]), 2, generator=g) - 0.5
    B = 4096
    x = torch.rand(B, 3, generator=g)
    G = torch.randn(B, 32, generator=g)
    return (gws, gas, gim), lay, offsets, table, x, G


# ------------------------------------------------------------------------------------------------ the reference's kernels
def _load(name):
    import importlib.util
    so = os.path.join(ROOT, "oracle", "_ref", name, name + ".so")
    if not os.path.exists(so):
        raise SystemExit(f"{so} not built: run oracle/build_ref.py first")
    spec = importlib.util.spec_from_file_location(name, so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_reference_kernels(oracle_ops):
    """Every output of the reference's kernels the pins compare, whole (CPU tensors), plus the digests of their inputs."""
    rm, ge, sh, fr = _load("_raymarching_face"), _load("_gridencoder"), _load("_shencoder"), _load("_freqencoder")
    r, meta = {}, {}
    # near/far + one marching round of 8 steps from the near plane
    sc, ro, rd = march_inputs()
    N = ro.shape[0]
    aabb, bits = sc.state["aabb_infer"], sc.state["density_bitfield"]
    meta["march"] = digest(ro, rd, aabb, bits)
    nears = torch.empty(N, device="cuda"); fars = torch.empty(N, device="cuda")
    rm.near_far_from_aabb(ro.cuda(), rd.cuda(), aabb.cuda(), N, 0.05, nears, fars)
    n_o, f_o = oracle_ops.near_far_from_aabb(ro, rd, aabb, 0.05)
    alive = torch.arange(N, dtype=torch.int32)
    M = oracle_ops.march_rays(N, 8, alive, n_o.clone(), ro, rd, 1.0, bits, 1, 128, n_o, f_o, 128, False, 1 / 256, 16)[0].shape[0]
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); deltas = torch.zeros(M, 2, device="cuda")
    rm.march_rays(N, 8, alive.cuda(), nears.clone(), ro.cuda(), rd.cuda(), 1.0, 1 / 256, 16, 1, 128, bits.cuda(), nears, fars, xyzs, dirs, deltas,
                  torch.zeros(N, device="cuda"))
    r.update(nears=nears, fars=fars, march_xyzs=xyzs, march_deltas=deltas)
    # inference compositing
    n_alive, n_step, alive, t, ws, dp, img, sig, rgb, dl = composite_inputs()
    meta["composite"] = digest(alive, t, ws, dp, img, sig, rgb, dl)
    dev = [x.clone().cuda() for x in (alive, t, ws, dp, img)]
    rm.composite_rays(n_alive, n_step, 0.01, dev[0], dev[1], sig.cuda(), rgb.cuda(), dl.cuda(), dev[2], dev[3], dev[4])
    r.update(comp_alive=dev[0], comp_t=dev[1], comp_ws=dev[2], comp_depth=dev[3], comp_image=dev[4])
    # grid encoder forward
    for D in (3, 2):
        lay, emb, x, off = grid_inputs(D)
        meta[f"grid{D}"] = digest(emb, x, off)
        out = torch.empty(16, 8192, 2, device="cuda")
        ge.grid_encode_forward(x.cuda(), emb.cuda(), off.cuda(), out, 8192, D, 2, 16, float(np.log2(lay.per_level_scale)), 16, None, 1, False, 0)
        r[f"grid{D}"] = out.permute(1, 0, 2).reshape(8192, 32)
    # SH + frequency encoders
    d, x = sh_freq_inputs()
    meta["sh_freq"] = digest(d, x)
    out = torch.empty(4096, 16, device="cuda")
    sh.sh_encode_forward(d.cuda(), out, 4096, 3, 4, None)
    o2 = torch.empty(2048, 42, device="cuda")
    fr.freq_encode_forward(x.cuda(), 2048, 2, 10, 42, o2)
    r.update(sh=out, freq=o2)
    # training-side: march_rays_train
    sc, ro, rd, nears, fars = train_rays(oracle_ops)
    bits = sc.state["density_bitfield"]
    meta["train_march"] = digest(ro, rd, nears, fars, bits)
    N, max_steps = ro.shape[0], 16
    M = N * max_steps
    xyzs, dirs, deltas = torch.zeros(M, 3, device="cuda"), torch.zeros(M, 3, device="cuda"), torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda")
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    rm.march_rays_train(ro.cuda(), rd.cuda(), bits.cuda(), 1.0, 1 / 256, max_steps, N, 1, 128, M, nears.cuda(), fars.cuda(), xyzs, dirs, deltas, rays, counter,
                        torch.zeros(N, device="cuda"))
    r.update(train_rays=rays, train_counter=counter, train_xyzs=xyzs, train_deltas=deltas)
    # training-side: compositing forward + backward
    rays_s, Ms, sig, rgb, amb, dl = segments()
    (gws, gas, gim), lay, offsets, table, x, G = train_grid_inputs()
    meta["train_composite"] = digest(rays_s, sig, rgb, amb, dl, gws, gas, gim)
    Ns = rays_s.shape[0]
    ws, asum, depth, image = [torch.empty(Ns, device="cuda") for _ in range(3)] + [torch.empty(Ns, 3, device="cuda")]
    rm.composite_rays_train_forward(sig.cuda(), rgb.cuda(), amb.cuda(), dl.cuda(), rays_s.cuda(), Ms, Ns, 1e-4, ws, asum, depth, image)
    gs, gr, ga = torch.zeros(Ms, device="cuda"), torch.zeros(Ms, 3, device="cuda"), torch.zeros(Ms, device="cuda")
    rm.composite_rays_train_backward(gws.cuda(), gas.cuda(), gim.cuda(), sig.cuda(), rgb.cuda(), amb.cuda(), dl.cuda(), rays_s.cuda(), ws, asum, image, Ms, Ns,
                                     1e-4, gs, gr, ga)
    r.update(tc_ws=ws, tc_depth=depth, tc_image=image, tc_gsig=gs, tc_grgb=gr, tc_gamb=ga)
    # training-side: grid encoder dy_dx, backward, total variation
    meta["train_grid"] = digest(offsets, table, x, G)
    B = x.shape[0]
    S = float(np.log2(lay.per_level_scale))
    grad = G.view(B, 16, 2).permute(1, 0, 2).contiguous().cuda()
    out_r, dy_r = torch.empty(16, B, 2, device="cuda"), torch.empty(B, 16 * 3 * 2, device="cuda")
    ge.grid_encode_forward(x.cuda(), table.cuda(), offsets.cuda(), out_r, B, 3, 2, 16, S, 16, dy_r, 1, False, 0)
    ge_r, gi_r = torch.zeros_like(table).cuda(), torch.zeros(B, 3, device="cuda")
    ge.grid_encode_backward(grad, x.cuda(), table.cuda(), offsets.cuda(), ge_r, B, 3, 2, 16, S, 16, dy_r, gi_r, 1, False, 0)
    tv_r = torch.zeros_like(table).cuda()
    ge.grad_total_variation(x.cuda(), table.cuda(), tv_r, offsets.cuda(), 0.5, B, 3, 2, 16, S, 16, 1, False)
    r.update(tg_dydx=dy_r, tg_table_grad=ge_r, tg_input_grad=gi_r, tg_tv=tv_r)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in r.items()}, {"input_sha256": meta, "device": torch.cuda.get_device_name(0)}


def pack(r, meta):
    """The stored golden: small outputs whole, large ones as a fixed sample (indices stored beside the values)."""
    z = {}
    z["nf_rays"] = sample(r["nears"].shape[0], 2048, 0)
    z["nears"], z["fars"] = r["nears"][z["nf_rays"]].numpy(), r["fars"][z["nf_rays"]].numpy()
    # marching: which rows the reference filled (all of them, as bits), positions of the filled rows of a sample of rays
    valid = (r["march_deltas"][:, 0] > 0).numpy()
    z["march_valid_bits"], z["march_rows"] = np.packbits(valid), np.int64(valid.size)
    n_rays = r["nears"].shape[0]
    ray_s = sample(n_rays, 512, 1)
    rows = (ray_s[:, None].astype(np.int64) * 8 + np.arange(8)).reshape(-1)
    rows = rows[valid[rows]]
    z["march_xyz_rows"], z["march_xyzs"] = rows.astype(np.int32), r["march_xyzs"][rows].numpy()
    for k in ("comp_alive", "comp_t", "comp_ws", "comp_depth", "comp_image"):
        z[k] = r[k].numpy()
    for D in (3, 2):
        z[f"grid{D}_rows"] = sample(8192, 192, 10 + D)
        z[f"grid{D}"] = r[f"grid{D}"][z[f"grid{D}_rows"]].numpy()
    z["sh_rows"] = sample(4096, 256, 20)
    z["sh"] = r["sh"][z["sh_rows"]].numpy()
    z["freq_rows"] = sample(2048, 128, 21)
    z["freq"] = r["freq"][z["freq_rows"]].numpy()
    # march_rays_train: sample count of every ray (in ray-id order), the counter, and the samples of a sample of rays
    rays = r["train_rays"]
    order = torch.argsort(rays[:, 0].long())
    rr = rays[order]
    z["train_counts"], z["train_counter"] = rr[:, 2].numpy().astype(np.int16), r["train_counter"].numpy()
    ids = sample(rays.shape[0], 128, 30)
    segs = [torch.arange(int(rr[n, 1]), int(rr[n, 1] + rr[n, 2])) for n in ids]
    idx = torch.cat(segs).long()
    z["train_seg_rays"], z["train_xyzs"], z["train_deltas"] = ids, r["train_xyzs"][idx].numpy(), r["train_deltas"][idx].numpy()
    # training compositing: forward for a sample of rays, backward for a sample of points
    z["tc_rays"] = sample(r["tc_ws"].shape[0], 512, 31)
    for k in ("tc_ws", "tc_depth", "tc_image"):
        z[k] = r[k][z["tc_rays"]].numpy()
    z["tc_points"] = sample(r["tc_gsig"].shape[0], 1024, 32)
    for k in ("tc_gsig", "tc_grgb", "tc_gamb"):
        z[k] = r[k][z["tc_points"]].numpy()
    # training grid: dy_dx / input grad for a sample of inputs, table grad / TV for a sample of table entries
    z["tg_rows"] = sample(r["tg_dydx"].shape[0], 64, 33)
    z["tg_dydx"] = r["tg_dydx"][z["tg_rows"]].numpy()
    z["tg_grad_rows"] = sample(r["tg_input_grad"].shape[0], 512, 34)
    z["tg_input_grad"] = r["tg_input_grad"][z["tg_grad_rows"]].numpy()
    z["tg_entries"] = sample(r["tg_table_grad"].numel(), 2048, 35)
    z["tg_table_grad"] = r["tg_table_grad"].reshape(-1)[z["tg_entries"]].numpy()
    z["tg_tv"] = r["tg_tv"].reshape(-1)[z["tg_entries"]].numpy()
    z["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    return z


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=OUT)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    from oracle import ops
    ops.build()
    r, meta = run_reference_kernels(ops)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    np.savez_compressed(a.out, **pack(r, meta))
    print(f"wrote {a.out} ({os.path.getsize(a.out)} bytes)")


if __name__ == "__main__":
    main()
