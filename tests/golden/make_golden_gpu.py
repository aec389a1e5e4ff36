"""Generate tests/golden/reference_gpu.npz by EXECUTING THE REFERENCE on a CUDA GPU.

What runs is the reference itself, built and staged into oracle/_ref/ by oracle/build_ref.py and loaded by
oracle/ref_harness.py: its `grid` CUDA extension compiled for sm_100a and its hot-path Python (render_helpers,
voxel_helpers, lidar, criterion, se3pose, lidarFrame), with its own classes.  Sampling noise and sort ties are pinned as in
ref_harness.pinned().  The scenarios are built by the functions the tests themselves use (tests/test_gpu_ops.py,
tests/test_gpu_dropin_reference.py), so the stored outputs are what those tests compare against.  Outputs larger than a few
thousand values are stored as a fixed, seeded sample of their rows or entries, together with the sampled indices.

Run:  python tests/golden/make_golden_gpu.py      (needs a GPU and oracle/_ref; writes tests/golden/reference_gpu.npz)
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import nerfloam_b200 as nl  # noqa: E402
from oracle import ref_harness as H  # noqa: E402
import test_gpu_dropin_reference as D  # noqa: E402
import test_gpu_ops as O  # noqa: E402
from util import golden, product_map  # noqa: E402

N_ISECT_ROWS, N_ICDF_ROWS, N_RENDER_ROWS, N_EMB, N_DEC = 512, 256, 128, 8192, 1024


def sample(n, k, seed):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, k), replace=False)).astype(np.int64)


def rows_of(t, rows):
    return t.cpu()[torch.from_numpy(rows)].numpy()


def bf16_bits(t):
    return t.detach().contiguous().view(torch.int16).cpu().numpy()


def kernels(ref, out):
    """svo_intersect and inverse_cdf_sampling of the compiled reference on the inputs of tests/test_gpu_ops.py."""
    z = golden("render.npz")
    vs = float(z["voxel_size"])
    m = product_map(z["vox"], vs, z["id2emb"], z["emb_bf16"])
    ro = torch.from_numpy(z["rays_o"]).cuda()[None].contiguous()
    rd = torch.from_numpy(z["rays_d"]).cuda()[None].contiguous()
    pts, ch = m["centres"].cuda()[None].contiguous(), m["structure"].cuda()[None].contiguous()
    batched = [t.reshape(-1, 20) for t in ref.grid.svo_intersect(*O.intersect_batched(ro, rd, pts, ch), vs, 20)]
    single = [t[0] for t in ref.grid.svo_intersect(ro, rd, pts, ch, vs, 20)]
    n = batched[0].shape[0]
    assert all(torch.equal(a, b[:n]) for a, b in zip(batched, single)), "per-ray results depend on the batching"
    rows = sample(n, N_ISECT_ROWS, 1)
    out.update(isect_rows=rows, isect_idx=rows_of(batched[0], rows), isect_min=rows_of(batched[1], rows), isect_max=rows_of(batched[2], rows))
    si, sd, sl = ref.grid.inverse_cdf_sampling(*O.inverse_cdf_inputs(z), -1.0)
    S = si.shape[-1]
    rows = sample(si.numel() // S, N_ICDF_ROWS, 2)
    out.update(icdf_rows=rows, icdf_idx=rows_of(si.reshape(-1, S), rows), icdf_depth=rows_of(sd.reshape(-1, S), rows),
               icdf_dist=rows_of(sl.reshape(-1, S), rows))


def loops(ref, out):
    """The reference's bundle_adjust_frames, track_frame and render_rays + Criterion on the scenarios of
    tests/test_gpu_dropin_reference.py."""
    scans, ms0, dec0 = D.state(ref, nl, table_rows=4_000_000)
    p0 = D.initial_poses(ref, scans)
    emb_idx = sample(ms0["voxel_vertex_emb"].numel(), N_EMB, 3)
    out.update(pose0=p0.numpy(), emb_shape=np.array(ms0["voxel_vertex_emb"].shape), emb_idx=emb_idx)
    for k, v in dec0.state_dict().items():
        out[f"dec_idx_{k}"] = sample(v.numel(), N_DEC, 4)
        out[f"dec0_{k}"] = v.flatten().cpu().numpy()[out[f"dec_idx_{k}"]]
    for tag, upd in (("ba_dec", True), ("ba_frozen", False)):
        ms, dec, fr = D.clone_ms(ms0), copy.deepcopy(dec0), D.frames(ref, scans, p0)
        torch.manual_seed(11)
        with H.pinned(ref):
            ref.orig["bundle_adjust_frames"](fr, ms["voxel_vertex_emb"], ms, dec, D.criterion(ref), update_decoder=upd, **D.BA_KW)
        torch.cuda.synchronize()
        out[f"{tag}_pose"] = torch.stack([f.pose.data.detach().cpu() for f in fr]).numpy()
        out[f"{tag}_emb_bf16"] = bf16_bits(ms["voxel_vertex_emb"].flatten()[torch.from_numpy(emb_idx).cuda()])
        for k, v in dec.state_dict().items():
            if upd:
                out[f"{tag}_dec_{k}"] = v.flatten().cpu().numpy()[out[f"dec_idx_{k}"]]
            else:
                assert torch.equal(v, dec0.state_dict()[k])

    scans, ms0, dec0 = D.state(ref, nl)
    f = D.track_frame_input(ref, scans, p0)
    torch.manual_seed(21)
    with H.pinned(ref):
        pose_r, hit_r = ref.orig["track_frame"](copy.deepcopy(f.pose), f, D.clone_ms(ms0), copy.deepcopy(dec0), D.criterion(ref), **D.TRACK_KW)
    hit = hit_r.cpu().numpy().astype(bool).reshape(-1)
    out.update(track_pose=pose_r.data.detach().cpu().numpy(), track_hit=np.packbits(hit), track_hit_len=np.int64(hit.size))

    ro, rd, P, Cn = D.render_inputs(scans)
    with H.pinned(ref):
        o = ref.orig["render_rays"](ro, rd, D.clone_ms(ms0), copy.deepcopy(dec0), *D.RENDER_ARGS, chunk_size=-1)
        loss, _ = D.criterion(ref)(o, P[None], Cn[None, :, None])
    valid = o["valid_mask"].cpu().numpy()
    rows = sample(valid.shape[0], N_RENDER_ROWS, 5)
    out.update(render_ray_mask=np.packbits(o["ray_mask"].view(-1).cpu().numpy()), render_valid_shape=np.array(valid.shape),
               render_valid=np.packbits(valid.reshape(-1)), render_rows=rows, render_z=rows_of(o["z_vals"], rows),
               render_sdf=rows_of(o["sdf"].detach(), rows), render_loss=np.float64(loss.item()))


if __name__ == "__main__":
    assert torch.cuda.is_available(), "the reference's kernels need a GPU"
    ref = H.load()
    out = {}
    kernels(ref, out)
    loops(ref, out)
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_gpu.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")
