"""Second oracle pin: the REFERENCE'S OWN CUDA kernels vs the C restatement oracle/native_ops.c, op by op.

The reference's kernels (compiled unmodified for sm_100a) ran on a B200 on the inputs built by oracle/make_ref_kernel_golden.py;
tests/golden/ref_kernels.npz holds what they returned (large outputs as a fixed sample, indices stored beside the values).
These tests rebuild the same inputs, check them against the digests stored with the outputs, and hold the C oracle to the
stored outputs: they need neither the reference nor a GPU.

What may differ and why (SURVEY.md H2/H6): nvcc contracts a*b+c into FMA in the reference build while the oracle is
unfused, and the reference uses __expf/__sinf.  So positions are compared exactly where the arithmetic is discrete-safe
and within tolerances elsewhere; rows whose occupancy decision flipped are COUNTED and bounded, never masked."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import make_ref_kernel_golden as rk

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.npz")


@pytest.fixture(scope="module")
def ref():
    z = np.load(GOLDEN)
    return z, json.loads(bytes(z["meta"]).decode())["input_sha256"]


def test_near_far_and_march_vs_reference_kernels(ref, oracle_ops):
    z, sha = ref
    sc, ro, rd = rk.march_inputs()
    N = ro.shape[0]
    aabb, bits = sc.state["aabb_infer"], sc.state["density_bitfield"]
    assert rk.digest(ro, rd, aabb, bits) == sha["march"], "inputs differ from the ones the stored outputs were computed on"
    n_ref, f_ref = oracle_ops.near_far_from_aabb(ro, rd, aabb, 0.05)
    nf = torch.from_numpy(z["nf_rays"]).long()
    nears, fars = torch.from_numpy(z["nears"]), torch.from_numpy(z["fars"])
    dn = (nears - n_ref[nf]).abs().max().item()
    print(f"near/far: max |reference kernel - C oracle| = {dn:.2e} over {nf.numel()} sampled rays")
    assert dn <= 1e-6 and (fars - f_ref[nf]).abs().max().item() <= 1e-6
    # one marching round of 8 steps from the near plane
    alive = torch.arange(N, dtype=torch.int32)
    n_step = 8
    x_o, d_o, l_o = oracle_ops.march_rays(N, n_step, alive, n_ref.clone(), ro, rd, 1.0, bits, 1, 128, n_ref, f_ref, 128, False, 1 / 256, 16)
    M = x_o.shape[0]
    assert int(z["march_rows"]) == M
    ref_valid = torch.from_numpy(np.unpackbits(z["march_valid_bits"], count=M).astype(bool))    # rows the reference filled
    same_rows = ref_valid == (l_o[:, 0] > 0)
    n_flip = int((~same_rows).sum())
    n_samples = int((l_o[:, 0] > 0).sum())
    # positions of the filled rows of a fixed sample of rays
    rows = torch.from_numpy(z["march_xyz_rows"]).long()
    xr = torch.from_numpy(z["march_xyzs"])
    both = l_o[rows, 0] > 0
    dpos = (xr[both] - x_o[rows][both]).abs().max().item()
    print(f"march: {n_samples} samples, rows whose validity differs (FMA-contraction cell flips): {n_flip}, "
          f"max |dpos| on common rows of {rows.numel()} sampled rows = {dpos:.2e}")
    assert n_samples > 5000
    assert n_flip <= max(4, n_samples // 2000)
    # a flipped occupancy decision shifts every later sample of that ray by one step; exclude those rays from the position bar
    per_ray_ok = same_rows[: N * n_step].view(N, n_step).all(1)
    okrows = per_ray_ok[rows // n_step] & both
    assert okrows.sum() > 100
    assert (xr[okrows] - x_o[rows][okrows]).abs().max().item() <= 2e-6


def test_composite_vs_reference_kernel(ref, oracle_ops):
    z, sha = ref
    n_alive, n_step, alive, t, ws, dp, img, sig, rgb, deltas = rk.composite_inputs()
    assert rk.digest(alive, t, ws, dp, img, sig, rgb, deltas) == sha["composite"]
    ref_ = [x.clone() for x in (alive, t, ws, dp, img)]
    oracle_ops.composite_rays(n_alive, n_step, ref_[0], ref_[1], sig, rgb, deltas, ref_[2], ref_[3], ref_[4], 0.01)
    dev = [torch.from_numpy(z[k]) for k in ("comp_alive", "comp_t", "comp_ws", "comp_depth", "comp_image")]
    same_alive = (dev[0] >= 0) == (ref_[0] >= 0)
    print(f"composite: rays whose alive flag differs: {int((~same_alive).sum())}; max |ws diff| = {(dev[2] - ref_[2]).abs().max().item():.2e} (reference uses __expf)")
    assert int((~same_alive).sum()) <= 2
    assert (dev[2] - ref_[2]).abs().max().item() <= 5e-6 and (dev[4] - ref_[4]).abs().max().item() <= 5e-6


@pytest.mark.parametrize("D", [3, 2])
def test_grid_encoder_vs_reference_kernel(ref, oracle_ops, D):
    z, sha = ref
    lay, emb, x, off = rk.grid_inputs(D)
    assert rk.digest(emb, x, off) == sha[f"grid{D}"]
    rows = torch.from_numpy(z[f"grid{D}_rows"]).long()
    refo = oracle_ops.grid_encode(x[rows].contiguous(), emb, off, lay.per_level_scale, 16, 1, False, 0)
    d = (torch.from_numpy(z[f"grid{D}"]) - refo).abs().max().item()
    print(f"grid D={D}: max |reference kernel - C oracle| = {d:.2e} over {rows.numel()} sampled inputs")
    # The reference kernel derives each level scale with the DEVICE exp2f (gridencoder.cu:137; <= 2 ulp, MUFU.EX2 based); the
    # oracle and libgfpp use the host libm exp2f.  A 1-ulp difference in a scale of ~2047 moves the finest-level sample
    # position by ~1e-4 cells, i.e. up to ~2e-4 in a feature for U(-0.5,0.5) tables.  Bounded here, documented in DESIGN.md.
    assert d <= 5e-4


def test_sh_and_freq_vs_reference_kernels(ref, oracle_ops):
    z, sha = ref
    d, x = rk.sh_freq_inputs()
    assert rk.digest(d, x) == sha["sh_freq"]
    sr = torch.from_numpy(z["sh_rows"]).long()
    assert (torch.from_numpy(z["sh"]) - oracle_ops.sh_encode(d[sr].contiguous(), 4)).abs().max().item() <= 1e-6
    fr = torch.from_numpy(z["freq_rows"]).long()
    dd = (torch.from_numpy(z["freq"]) - oracle_ops.freq_encode(x[fr].contiguous(), 10)).abs()
    print(f"freq: max |reference(__sinf) - oracle(sinf)| = {dd.max().item():.2e} at arguments up to 2^9*0.8 rad")
    # the reference's __sinf loses accuracy at large arguments (SURVEY H6); low frequencies must agree tightly
    assert dd[:, :14].max().item() <= 5e-6 and dd.max().item() <= 5e-3
