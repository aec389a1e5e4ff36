"""Run the UNMODIFIED reference hot path on the GPU beside the product (test / baseline infrastructure only).

What this loads is the reference itself, staged by oracle/build_ref.py into the git-ignored oracle/_ref/:
  * oracle/_ref/grid/grid_ref.so  -- third_party/sparse_voxels compiled for sm_100a from the sources where they lie;
  * oracle/_ref/src/...           -- the reference's hot-path Python files, byte for byte (render_helpers.py,
                                     voxel_helpers.py, lidar.py, criterion.py, se3pose.py, lidarFrame.py, sample_util.py).
Nothing here is imported by the product (nerf-loam_b200/); callers are tests/, and bench.py's baseline legs.

The only thing restated here is the ~20 lines of tensor glue of Mapping.get_embeddings / update_grid_features
(src/mapping.py:294-339) that build the `map_states` dict -- mapping.py itself imports open3d / the data loaders and is
not importable -- including the reference's duplicate-row allocation and its [N,1] int32 CPU `voxel_id2embedding_id` table.
"""
import contextlib
import importlib
import importlib.util
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
SRC = os.path.join(REF_DIR, "src")
GRID_SO = os.path.join(REF_DIR, "grid", "grid_ref.so")

_loaded = None


def available():
    return os.path.exists(GRID_SO) and os.path.exists(os.path.join(SRC, "variations", "render_helpers.py"))


def load():
    """Import the staged reference modules with `grid` bound to the compiled reference extension.  Returns a namespace with
    the modules and the ORIGINAL functions (saved before any dropin.install() rebinding)."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("reference not staged: run `python oracle/build_ref.py` where /root/reference exists")
    spec = importlib.util.spec_from_file_location("grid_ref", GRID_SO)
    grid_ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(grid_ref)
    prev = sys.modules.get("grid")
    sys.modules["grid"] = grid_ref                     # `import grid as _ext` (voxel_helpers.py:22) binds at import time
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    VH = importlib.import_module("variations.voxel_helpers")
    RH = importlib.import_module("variations.render_helpers")
    lidar = importlib.import_module("variations.lidar")
    crit = importlib.import_module("criterion")
    se3 = importlib.import_module("se3pose")
    lf = importlib.import_module("lidarFrame")
    if prev is not None:
        sys.modules["grid"] = prev
    assert VH._ext is grid_ref
    ns = types.SimpleNamespace(grid=grid_ref, VH=VH, RH=RH, lidar=lidar, Decoder=lidar.Decoder, Criterion=crit.Criterion,
                               OptimizablePose=se3.OptimizablePose, LidarFrame=lf.LidarFrame, src=SRC,
                               orig={k: getattr(RH, k) for k in ("render_rays", "bundle_adjust_frames", "track_frame", "get_scores",
                                                                  "ray_sample", "ray_intersect")})
    _loaded = ns
    return ns


@contextlib.contextmanager
def pinned(ns, deterministic=True, stable_sort=True):
    """Context in which the reference's ORIGINAL functions are bound in its module and its two unspecified behaviours are
    pinned like the goldens pin them (tests/golden/make_golden.py): sampler noise constant 0.5 (ray_sample(..., fixed=True),
    voxel_helpers.py:298-299) and torch.sort ties in DFS order (stable=True; voxel_helpers.py:546 leaves them to an unstable
    sort).  Everything else is the reference as shipped."""
    RH, VH = ns.RH, ns.VH
    saved = {k: getattr(RH, k) for k in ns.orig}
    saved_sort = torch.Tensor.sort
    for k, v in ns.orig.items():
        setattr(RH, k, v)
    if deterministic:
        RH.ray_sample = lambda inter, step_size=0.01, fixed=False: VH.ray_sample(inter, step_size=step_size, fixed=True)
    if stable_sort:
        torch.Tensor.sort = lambda self, dim=-1, descending=False, stable=True: saved_sort(self, stable=True, dim=dim, descending=descending)
    try:
        yield ns
    finally:
        torch.Tensor.sort = saved_sort
        for k, v in saved.items():
            setattr(RH, k, v)


def reference_map_states(voxels, children, features, voxel_size, table_rows=None, init_std=0.0, seed=0, device="cuda"):
    """src/mapping.py:320-339 + :294-317 on the three CPU tensors of svo.get_centres_and_children():
    map_states dict in the reference's exact format (CPU index tensors, CUDA bf16 leaf table requiring grad, [N,1] int32 CPU
    voxel_id2embedding_id; rows allocated once per *reference* to a new vertex, duplicates included).  table_rows: size of
    the id table (the reference allocates 2e9 rows = 8 GB, mapping.py:76; any size > max vertex id behaves identically)."""
    centres = ((voxels[:, :3] + voxels[:, -1:] / 2) * voxel_size).float()
    structure = torch.cat([children, voxels[:, -1:]], -1).int()
    n = voxels.shape[0]
    id2 = -torch.ones((int(table_rows or n), 1), dtype=torch.int)
    flat = features.reshape(-1).long()
    valid = flat[flat.ne(-1)]
    existence = torch.nn.functional.embedding(valid, id2)
    add = valid[existence.eq(-1).view(-1)]
    emb = torch.zeros((add.shape[0], 16), dtype=torch.bfloat16)
    if init_std > 0:
        # one value per VERTEX (not per row): duplicate rows of a vertex get the same value, so the run does not depend on
        # which duplicate wins the racy index_put_ (SURVEY A.1)
        g = torch.Generator().manual_seed(seed)
        per_vertex = (torch.randn((n, 16), generator=g) * init_std).to(torch.bfloat16)
        emb = per_vertex[add].contiguous()
    # `add` repeats a vertex once per voxel that references it, so which of its rows the table keeps is unspecified (a racy
    # index_put_ in the reference, and a multi-threaded one on the host here): pinned to the last, so that every process builds
    # the same table and row-wise results recorded in one process hold in another
    last = torch.full((id2.shape[0],), -1, dtype=torch.long).scatter_reduce_(0, add, torch.arange(add.shape[0]), reduce="amax")
    id2[add] = last[add].int().view(-1, 1)
    centres.requires_grad_()
    return {"voxel_vertex_idx": features, "voxel_center_xyz": centres, "voxel_structure": structure,
            "voxel_vertex_emb": emb.to(device).requires_grad_(), "voxel_id2embedding_id": id2}


def args(max_depth=40.0, trunc=0.3, fs_weight=1, sdf_weight=10000.0):
    """The slice of the parsed YAML that Criterion reads (criterion.py:7-14)."""
    return types.SimpleNamespace(criteria={"eiko_weight": 0.1, "sdf_weight": sdf_weight, "fs_weight": fs_weight, "sdf_truncation": trunc},
                                 data_specs={"max_depth": max_depth})
