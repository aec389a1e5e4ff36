"""The drop-in boundary against the REFERENCE'S OWN loop on the B200 (SURVEY.md section 8 b-4).

tests/golden/reference_gpu.npz holds what the unmodified reference computed on a B200 for the scenarios below: its own
bundle_adjust_frames / track_frame / render_rays (render_helpers.py:321-514: eager PyTorch + its compiled `grid` extension +
autograd + torch.optim.Adam), run with its own classes -- Criterion, LidarFrame, OptimizablePose, Decoder -- on a `map_states`
dict in mapping.py's exact format (CPU index tensors, [N,1] int32 voxel_id2embedding_id, duplicate-row bf16 CUDA leaf table),
with the sampling noise and sort ties pinned (oracle/ref_harness.pinned).  tests/golden/make_golden_gpu.py regenerates it with
the scenario builders of this module.  These tests run the functions `nerfloam_b200.dropin.install()` binds in the reference's
place on identical inputs and seeds, and compare the parameters after 3 optimiser steps.  Outputs larger than a few thousand
values are stored as a fixed, seeded sample of their entries.
"""
import copy
import importlib
import sys
import types

import numpy as np
import pytest
import torch

from util import bf16_from_bits, golden

pytestmark = pytest.mark.gpu

VS, MD, TR = 0.3, 40.0, 0.3          # configs/kitti/kitti.yaml
LR = [0.01, 0.005, 0.001]
BA_KW = dict(voxel_size=VS, step_size=0.5 * VS, N_rays=1024, num_iterations=3, truncation=TR, max_voxel_hit=20, max_distance=MD,
             learning_rate=LR, update_pose=True)
TRACK_KW = dict(voxel_size=VS, N_rays=1024, step_size=0.2 * VS, num_iterations=3, truncation=TR, learning_rate=0.06, max_voxel_hit=20,
                max_distance=MD, depth_variance=True)
RENDER_ARGS = (0.5 * VS, VS, TR, 20, MD)


def scene(nl, n_scans=3):
    syn = nl.synthetic
    scans = [syn.make_scan(n_beams=32, n_az=600, seed=100 + i, sensor_xyz=(1.0 * i, 0.1 * i, 0.0), yaw=0.02 * i) for i in range(n_scans)]
    o = nl.svo.Octree()
    o.init(256 * 256 * 4, 16, VS)
    for pts, cos, pose in scans:
        o.insert(torch.from_numpy(syn.voxelize(pts, pose, VS)))
    return scans, o.get_centres_and_children()


def initial_poses(cls, scans):
    """6-vector poses of the scans, frames 1.. perturbed (seeded)."""
    g = torch.Generator().manual_seed(5)
    out = []
    for i, (pts, cos, pose) in enumerate(scans):
        p6 = cls.OptimizablePose.from_matrix(torch.from_numpy(pose.copy())).data.detach().clone()
        if i > 0:
            p6 = p6 + torch.cat([torch.randn(3, generator=g) * 0.02, torch.randn(3, generator=g) * 0.002])
        out.append(p6.float())
    return torch.stack(out)


def frames(cls, scans, poses):
    """LidarFrame / OptimizablePose objects of `cls` (lidarFrame.py:10-25 with new_keyframe=True adopts the pose object).  The scan
    tensors are device-resident: the reference indexes `frame.rays_d` with a CUDA mask (render_helpers.py:371-372), which torch >= 2
    rejects for CPU tensors."""
    return [cls.LidarFrame(i, torch.from_numpy(pts).cuda(), torch.from_numpy(cos).cuda(), cls.OptimizablePose(poses[i].clone()), new_keyframe=True)
            for i, (pts, cos, _) in enumerate(scans)]


def track_frame_input(cls, scans, poses):
    f = frames(cls, scans, poses)[1]
    f.index = 5                                                # lr/3 branch of render_helpers.py:448-450
    return f


def state(cls, nl, table_rows=None):
    from oracle import ref_harness as H
    scans, (voxels, children, features) = scene(nl)
    ms = H.reference_map_states(voxels, children, features, VS, table_rows=table_rows, init_std=0.01, seed=3)
    torch.manual_seed(777)
    dec = cls.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).cuda()
    return scans, ms, dec


def criterion(cls):
    from oracle import ref_harness as H
    return cls.Criterion(H.args(MD, TR))


def clone_ms(ms):
    out = dict(ms)
    out["voxel_vertex_emb"] = ms["voxel_vertex_emb"].detach().clone().requires_grad_()
    return out


def render_inputs(scans):
    """2048 seeded rays of scan 0 in the world frame: (rays_o, rays_d, points, cosines)."""
    pts, cos, pose = scans[0]
    sel = np.sort(np.random.default_rng(0).choice(pts.shape[0], 2048, replace=False))
    P, Cn = torch.from_numpy(pts[sel]).cuda(), torch.from_numpy(cos[sel]).cuda()
    T = torch.from_numpy(pose).cuda()
    rd = ((P / (P.norm(dim=-1, keepdim=True) + 1e-8)) @ T[:3, :3].T)[None].contiguous()
    ro = T[:3, 3].reshape(1, 1, 3).expand_as(rd).contiguous()
    return ro, rd, P, Cn


@pytest.fixture(scope="module")
def nl():
    import nerfloam_b200 as nl
    assert torch.cuda.is_available()
    return nl


@pytest.fixture(scope="module")
def cls(nl):
    return types.SimpleNamespace(LidarFrame=nl.frame.LidarFrame, OptimizablePose=nl.se3pose.OptimizablePose, Decoder=nl.lidar.Decoder,
                                 Criterion=nl.criterion.Criterion)


@pytest.fixture(scope="module")
def gold():
    return golden("reference_gpu.npz")


@pytest.fixture(scope="module")
def rebound(nl, tmp_path_factory):
    """The reference's `variations.render_helpers` module after dropin.install(): a stand-in with the reference's module layout
    (its sources are not part of this repository) on the path given to install(), whose functions must come back rebound."""
    src = tmp_path_factory.mktemp("reference_src")
    (src / "variations").mkdir()
    (src / "variations" / "__init__.py").write_text("")
    (src / "variations" / "render_helpers.py").write_text(
        "".join(f"def {n}(*args, **kwargs):\n    raise NotImplementedError\n" for n in ("render_rays", "bundle_adjust_frames", "track_frame", "get_scores")))
    (src / "variations" / "lidar.py").write_text("class Decoder:\n    pass\n")
    import nerfloam_b200.dropin as dropin
    dropin.install(reference_src=str(src))
    rh = importlib.import_module("variations.render_helpers")
    for name in ("render_rays", "bundle_adjust_frames", "track_frame", "get_scores"):
        assert getattr(rh, name) is getattr(nl.render_helpers, name)          # what mapping.py:179 / tracking.py now call
    assert importlib.import_module("variations.lidar").Decoder is nl.lidar.Decoder
    yield rh
    sys.path.remove(str(src))
    for name in ("variations", "variations.render_helpers", "variations.lidar"):
        sys.modules.pop(name, None)


def test_reference_inputs_are_reproduced(nl, cls, gold):
    """The scenario's inputs built here equal the reference's own: initial poses (from_matrix + perturbation) and the decoder
    initialisation under the same seed (sampled entries)."""
    scans, ms0, dec0 = state(cls, nl)
    np.testing.assert_array_equal(initial_poses(cls, scans).numpy(), gold["pose0"])
    assert tuple(ms0["voxel_vertex_emb"].shape) == tuple(gold["emb_shape"])
    for k, v in dec0.state_dict().items():
        np.testing.assert_array_equal(v.flatten().cpu().numpy()[gold[f"dec_idx_{k}"]], gold[f"dec0_{k}"])


@pytest.mark.parametrize("update_decoder", [True, False])
def test_bundle_adjust_frames_reference_objects_through_dropin(nl, cls, gold, rebound, update_decoder):
    scans, ms0, dec0 = state(cls, nl, table_rows=4_000_000)
    p_0 = torch.from_numpy(gold["pose0"])
    tag = "ba_dec" if update_decoder else "ba_frozen"
    ms_p, dec_p, fr_p = clone_ms(ms0), copy.deepcopy(dec0), frames(cls, scans, p_0)
    torch.manual_seed(11)
    rebound.bundle_adjust_frames(fr_p, ms_p["voxel_vertex_emb"], ms_p, dec_p, criterion(cls), deterministic=True, ray_selection="host",
                                 update_decoder=update_decoder, **BA_KW)
    torch.cuda.synchronize()

    # poses: frame 0 frozen, the others moved and agree
    p_r = torch.from_numpy(gold[f"{tag}_pose"])
    p_p = torch.stack([f.pose.data.detach().cpu() for f in fr_p])
    assert torch.equal(p_p[0], p_0[0]) and torch.equal(p_r[0], p_0[0])
    assert float((p_r[1:] - p_0[1:]).abs().max()) > 1e-3
    # 3 Adam steps of lr 1e-3: the first step moves every coordinate by exactly +-lr, so agreement to a small fraction of lr
    # means the gradient signs and the later normalised steps agree
    np.testing.assert_allclose(p_p.numpy(), p_r.numpy(), atol=1e-4)
    # decoder: Adam moves every element by ~lr per step whatever the size of its gradient, so an element whose gradient is numerically
    # zero (its sign is rounding noise on BOTH sides) may legitimately differ by a fraction of lr: all but a sliver agree to 2e-4
    # (4 % of one step), none by more than a step
    lr_dec = LR[1]
    for k, a in dec_p.state_dict().items():
        if update_decoder:
            idx = torch.from_numpy(gold[f"dec_idx_{k}"]).long()
            a0, a = dec0.state_dict()[k].flatten().cpu()[idx], a.flatten().cpu()[idx]
            b = torch.from_numpy(gold[f"{tag}_dec_{k}"])
            assert float((b - a0).abs().max()) > 1e-3
            d = (a - b).abs()
            assert float((d > 2e-4).float().mean()) < 5e-3 and float(d.max()) < lr_dec, (k, float((d > 2e-4).float().mean()), float(d.max()))
        else:
            assert torch.equal(a, dec0.state_dict()[k])
    # embeddings (bf16, same row numbering: both sides use the reference's table).  The update as a whole agrees (norm-wise), the
    # same entries moved, and only a sliver of entries differs by more than a fifth of one Adam step
    idx = torch.from_numpy(gold["emb_idx"]).long()
    e_0, e_p = (t["voxel_vertex_emb"].detach().float().cpu().flatten()[idx] for t in (ms0, ms_p))
    e_r = bf16_from_bits(gold[f"{tag}_emb_bf16"]).float()
    u_r, u_p = e_r - e_0, e_p - e_0
    moved_r, moved_p = u_r.abs() > 1e-3, u_p.abs() > 1e-3
    stats = dict(moved_ref=float(moved_r.float().mean()), moved_ours=float(moved_p.float().mean()),
                 both=float((moved_r & moved_p).float().sum() / moved_r.float().sum()),
                 update_rel=float((u_p - u_r).norm() / u_r.norm()), frac_gt_2e3=float(((e_p - e_r).abs() > 2e-3).float().mean()),
                 max_abs=float((e_p - e_r).abs().max()))
    print("embedding update, drop-in vs reference:", stats)
    assert stats["moved_ref"] > 0.01
    assert stats["update_rel"] < 0.05, stats
    assert stats["frac_gt_2e3"] < 5e-3, stats


@pytest.mark.parametrize("impl", ["simt", "tc"])
def test_track_frame_reference_objects_through_dropin(nl, cls, gold, rebound, impl, monkeypatch):
    """Three tracking iterations, reference vs drop-in.  The pose gradient of a nearly converged pose is a sum of ~2e4 per-sample
    terms that cancel to ~1e-4 of their absolute sum, so it amplifies every rounding difference by ~1e4:
      * with the fp32 CUDA-core decoder (NL_MLP_IMPL=simt) the drop-in reproduces the reference's poses to 2e-5 -- the fused
        pipeline itself (traversal, sampling, gather, loss, pose Jacobian, Adam) is exact;
      * with the tensor-core decoder (default) the 3xTF32 products are exact to 2^-22 but the tensor core ACCUMULATES with
        truncation, a coherent ~1e-6 relative error per pre-activation, which this gradient turns into ~1e-3 (measured against an
        fp64 run: 1.1e-3 vs 1e-5 for fp32 FMA) and three Adam steps into <= 5 % of a step.  Mapping gradients (no such
        cancellation) meet 1e-4 with the same kernels (test_single_iteration_gradients_vs_oracle_autograd)."""
    monkeypatch.setenv("NL_MLP_IMPL", impl)
    scans, ms0, dec0 = state(cls, nl)
    f_p = track_frame_input(cls, scans, torch.from_numpy(gold["pose0"]))
    pose_in = f_p.pose.data.detach().clone()
    torch.manual_seed(21)
    pose_p, hit_p = rebound.track_frame(copy.deepcopy(f_p.pose), f_p, clone_ms(ms0), copy.deepcopy(dec0), criterion(cls), deterministic=True,
                                        ray_selection="host", **TRACK_KW)
    assert type(pose_p).__name__ == "OptimizablePose" and pose_p.data.is_cuda
    assert hit_p is not None
    hit_r = np.unpackbits(gold["track_hit"])[:int(gold["track_hit_len"])].astype(bool)
    assert np.array_equal(hit_p.cpu().numpy().reshape(-1), hit_r)
    pose_r = torch.from_numpy(gold["track_pose"])
    assert float((pose_r - pose_in).abs().max()) > 1e-3
    lr = 0.06 / 3
    d = (pose_p.data.detach().cpu() - pose_r).abs()
    print(f"track_frame drop-in vs reference ({impl}): max |pose diff| = {float(d.max()):.2e} (rotation {float(d[3:].max()):.2e}), lr = {lr}")
    # translation entries are ~2000 (+2000 m offset): their fp32 resolution is 1.2e-4, so only the rotation part is informative
    assert float(d[3:].max()) < (2e-5 if impl == "simt" else 0.05 * lr)
    assert float(d[:3].max()) < 1e-3


def test_render_rays_and_criterion_reference_objects(nl, cls, gold):
    """render_rays through the drop-in feeding Criterion.forward: same loss, same ray mask and sample layout as the reference's own
    render_rays + Criterion."""
    scans, ms0, dec0 = state(cls, nl)
    ro, rd, P, Cn = render_inputs(scans)
    out_p = nl.render_helpers.render_rays(ro, rd, clone_ms(ms0), copy.deepcopy(dec0), *RENDER_ARGS, chunk_size=-1, deterministic=True)
    loss_p, _ = criterion(cls)(out_p, P[None], Cn[None, :, None])
    ray_mask = np.unpackbits(gold["render_ray_mask"])[:P.shape[0]].astype(bool)
    assert np.array_equal(out_p["ray_mask"].view(-1).cpu().numpy(), ray_mask)
    valid = out_p["valid_mask"].cpu().numpy()
    assert valid.shape == tuple(gold["render_valid_shape"])
    assert np.array_equal(np.packbits(valid.reshape(-1)), gold["render_valid"])
    rows = gold["render_rows"]
    np.testing.assert_allclose(out_p["z_vals"].cpu().numpy()[rows], gold["render_z"], rtol=2e-6)
    np.testing.assert_allclose(out_p["sdf"].detach().cpu().numpy()[rows], gold["render_sdf"], atol=1e-5)
    np.testing.assert_allclose(float(loss_p), float(gold["render_loss"]), rtol=1e-5)
