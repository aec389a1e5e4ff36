"""Shared helpers for the tests (golden loading, map construction through the product API)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
G = os.path.join(ROOT, "tests", "golden")


def golden(name):
    return np.load(os.path.join(G, name))


def bf16_from_bits(a):
    return torch.from_numpy(a.copy()).view(torch.bfloat16)


def product_map(vox, voxel_size, id2emb=None, emb_bits=None, device="cuda", grid_dim=256 * 256 * 4):
    """Octree + MapState through the product code (svo.Octree.export_map + engine.MapState)."""
    import nerfloam_b200 as nl
    o = nl.svo.Octree()
    o.init(grid_dim, 16, voxel_size)
    o.insert(torch.from_numpy(np.ascontiguousarray(vox, np.int32)))
    centres, structure, vertex = o.export_map()
    out = {"octree": o, "centres": centres, "structure": structure, "vertex": vertex}
    if id2emb is not None:
        v = vertex.long()
        flat = torch.from_numpy(id2emb.reshape(-1)).long()
        rows = torch.where(v >= 0, flat[v.clamp(min=0)], torch.full_like(v, -1)).int()
        out["vox2row"] = rows
        if emb_bits is not None:
            emb = bf16_from_bits(emb_bits).to(device)
            out["state"] = nl.engine.MapState(centres, structure, rows, emb, device)
    return out


def load_decoder(z, prefix, device="cuda", width=256):
    import nerfloam_b200 as nl
    dec = nl.lidar.Decoder(depth=2, width=width, in_dim=16, skips=[], embedder="none", multires=0)
    sd = {k[len(prefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix)}
    dec.load_state_dict(sd)
    return dec.to(device)


class Args:
    def __init__(self, max_depth=40.0, trunc=0.3):
        self.criteria = {"eiko_weight": 0.1, "sdf_weight": 10000.0, "fs_weight": 1, "sdf_truncation": trunc}
        self.data_specs = {"max_depth": max_depth}
