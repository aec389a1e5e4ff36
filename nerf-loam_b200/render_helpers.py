"""Drop-in for src/variations/render_helpers.py: render_rays (:190), bundle_adjust_frames (:321),
track_frame (:428), get_scores (:97) with the reference signatures, running on the fused sm_100a kernel
chain (engine.SDFEngine) instead of ~60 eager PyTorch ops + 2 CUDA kernels + autograd per iteration.

Behavioural notes (also in DESIGN.md):
  * ray/voxel intersection order for hits with bit-identical min_depth is the DFS emission order (the
    reference leaves it to an unstable torch.sort);
  * stochastic sampling noise comes from a counter-based generator inside the kernel seeded from torch's
    global generator (the reference draws a data-dependent-shaped uniform_() tensor); pass
    deterministic=True or noise=<tensor> for bit-reproducible sampling against the reference;
  * `max_voxel_hit` and render_rays' `truncation` are accepted and ignored exactly like the reference
    (voxel_helpers.py:531-533; render_helpers.py:190-318);
  * the unused autograd.grad(sdf, xyz) of render_helpers.py:293-297 is not computed.
"""
import os
import weakref
from copy import deepcopy

import torch

from . import _capi
from .engine import DecoderBuffers, FusedAdam, MapState, SDFEngine, alloc_act, mlp_forward, mlp_train

MAX_DEPTH = 80.0
# initial sample capacity per ray of the fused loops (measured averages: ~10.5 mapping, ~19 tracking on the KITTI-shape scan); a call
# that exceeds it is undone and redone with a larger engine (bundle_adjust_frames / track_frame below), never silently truncated
SAMPLES_PER_RAY_MAP = 40
SAMPLES_PER_RAY_TRACK = 64

_ENGINES = {}


def _engine(n_rays, min_samples, device):
    """Engines are cached by capacity class (power-of-two rays / samples)."""
    r = 1 << max(10, (int(n_rays) - 1).bit_length())
    m = 1 << max(16, (int(min_samples) - 1).bit_length())
    key = (r, m, str(device))
    e = _ENGINES.get(key)
    if e is None:
        for k in [k for k in _ENGINES if k[0] <= r and k[1] <= m and k[2] == str(device)]:
            del _ENGINES[k]
        e = _ENGINES[key] = SDFEngine(r, m, device)
    return e


def _seed_from_torch():
    return int(torch.randint(1, 2 ** 31 - 1, (1,)).item())


def _cfg(step_size, voxel_size, max_distance, crit=None):
    """Kernel configuration.  `crit` is duck-typed on the attributes src/criterion.py:7-14 sets (truncation, fs_weight,
    sdf_weight, max_dpeth (sic)), so the reference's own Criterion instance works as well as nerfloam_b200's."""
    c = dict(step_size=float(step_size), voxel_size=float(voxel_size), max_distance=float(max_distance))
    if crit is not None:
        c.update(truncation=float(crit.truncation), max_depth=float(crit.max_dpeth), fs_weight=float(crit.fs_weight),
                 sdf_weight=float(crit.sdf_weight))
    return c


def _run_with_capacity(fn, n_rays, device, samples_per_ray=40):
    """Run fn(engine) and grow the sample capacity if the kernels report it was exceeded."""
    cap = n_rays * samples_per_ray
    while True:
        eng = _engine(n_rays, cap, device)
        fn(eng)
        st = eng.read_stats()
        if st.error & 4:
            _check_ctl([4], "render_rays")
        if st.error & 2:
            cap = max(cap * 2, st.n_samples + 1)
            continue
        return eng, st


class _RenderSDF(torch.autograd.Function):
    """Attaches the autograd graph to the SDF values the fused forward already produced: sdf of the valid
    samples as a differentiable function of (rays_o, rays_d, embeddings, decoder params).  backward runs
    the fused MLP backward (forward recomputed in-kernel), the gather backward and the ray chain rule."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, emb, pack, *dec_params):
        ctx.pack = pack
        return pack["sdf"]

    @staticmethod
    def backward(ctx, gsdf):
        import ctypes as C
        s = ctx.pack
        m, dec_mod, cfg = s["m"], s["dec"], s["cfg"]
        M = s["xyz"].shape[0]
        dev = s["xyz"].device
        bufs = DecoderBuffers.of(dec_mod, dev)
        bufs.refresh_transposes()
        bufs.gradflat.zero_()
        need_dec = any(ctx.needs_input_grad[4:])
        W = bufs.width
        sdf = torch.empty(M, dtype=torch.float32, device=dev)
        dfeats = torch.empty((M, 16), dtype=torch.float32, device=dev)
        act = alloc_act(W, M, dev) if need_dec else None
        g = gsdf.contiguous().float()
        lib, st = _capi.lib(), _capi.stream_ptr()
        mlp_train(bufs, M, None, s["feats"], sdf, dfeats, need_dec, act, dsdf_ext=g)
        need_emb = ctx.needs_input_grad[2]
        need_rays = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        grad_emb = torch.zeros((m.emb.shape[0], 16), dtype=torch.float32, device=dev) if need_emb else None
        dxyz = torch.empty((M, 3), dtype=torch.float32, device=dev) if need_rays else None
        if need_emb or need_rays:
            _capi.check(lib.nl_gather_trilinear_bwd(M, None, _capi.ptr(s["xyz"]), _capi.ptr(s["vox"]), _capi.ptr(m.centres),
                                                    _capi.ptr(m.vox2row), _capi.ptr(m.emb), float(cfg["voxel_size"]),
                                                    _capi.ptr(dfeats), 1, _capi.ptr(grad_emb), _capi.ptr(dxyz), None, None, None,
                                                    None, 0, None, st), "nl_gather_trilinear_bwd")
            _capi.LAUNCHES += 1
        g_o = g_d = None
        if need_rays:  # xyz = o + d * depth
            ray = s["ray"].long()
            g_o = torch.zeros((s["R"], 3), dtype=torch.float32, device=dev).index_add_(0, ray, dxyz)
            g_d = torch.zeros((s["R"], 3), dtype=torch.float32, device=dev).index_add_(0, ray, dxyz * s["depth"].unsqueeze(-1))
        dec_grads = [t.clone() for t in bufs.grads] if need_dec else [None] * 6      # own copies: the buffers are cached per decoder
        return (g_o, g_d, grad_emb.to(m.emb.dtype) if need_emb else None, None, *dec_grads)


def _decoder_params(dec):
    return [dec.pts_linears[0].weight, dec.pts_linears[0].bias, dec.pts_linears[1].weight, dec.pts_linears[1].bias,
            dec.sdf_out.weight, dec.sdf_out.bias]


def render_rays(rays_o, rays_d, map_states, sdf_network, step_size, voxel_size, truncation, max_voxel_hit, max_distance,
                chunk_size=10000, profiler=None, return_raw=False, deterministic=False, noise=None, reference_compat=True):
    """render_helpers.py:190-318.  rays_o / rays_d: [1,R,3] CUDA fp32.  Returns the reference's dict
    (z_vals [R_hit,S_max], sdf, ray_mask [1,R], valid_mask, sampled_xyz) or None when nothing is hit.
    The result is differentiable w.r.t. rays, embeddings and decoder parameters like the reference's."""
    dev = rays_o.device
    if dev.type != "cuda":
        raise RuntimeError("render_rays runs on the GPU only (no CPU fallback)")
    if profiler is not None:
        profiler.tick("ray_intersect")
    ro = rays_o.reshape(-1, 3).float().contiguous()
    rd = rays_d.reshape(-1, 3).float().contiguous()
    R = ro.shape[0]
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    emb_in = m.emb if isinstance(map_states, MapState) else map_states["voxel_vertex_emb"]
    if not (emb_in.is_cuda and emb_in.dtype == torch.bfloat16):
        emb_in = m.emb
    cfg = _cfg(step_size, voxel_size, max_distance)
    seed = 0 if (deterministic or noise is not None) else _seed_from_torch()
    bufs = DecoderBuffers.of(sdf_network, dev)
    with torch.no_grad():
        eng, st = _run_with_capacity(lambda e: e.forward(m, bufs, R, cfg, ro.detach(), rd.detach(), noise, seed, reference_compat),
                                     R, dev)
    if profiler is not None:
        profiler.tok("ray_intersect")
    if st.n_hit_rays <= 0 or (st.error & 1) or st.n_samples == 0:
        return None
    M, Rh, S = st.n_samples, st.n_hit_rays, st.max_samples
    pack = dict(xyz=eng.s_xyz[:M].clone(), vox=eng.s_vox[:M].clone(), ray=eng.s_ray[:M].clone(), depth=eng.s_depth[:M].clone(),
                feats=eng.feats[:M].clone(), sdf=eng.sdf[:M].clone(), m=m, dec=sdf_network, cfg=cfg, R=R)
    sdf_valid = _RenderSDF.apply(ro, rd, emb_in, pack, *_decoder_params(sdf_network))
    ray = pack["ray"].long()
    row = eng.hit_rank[:R].long()[ray]
    col = torch.arange(M, device=dev) - eng.ray_offset[:R].long()[ray]
    z_vals = torch.full((Rh, S), MAX_DEPTH, dtype=torch.float32, device=dev)
    z_vals[row, col] = pack["depth"]
    valid = torch.zeros((Rh, S), dtype=torch.bool, device=dev)
    valid[row, col] = True
    sdf = torch.ones((Rh, S), dtype=torch.float32, device=dev).index_put((row, col), sdf_valid)
    return {"z_vals": z_vals, "sdf": sdf, "ray_mask": (eng.hit_rank[:R] >= 0).view(1, -1), "valid_mask": valid,
            "sampled_xyz": pack["xyz"]}


def _lattice_offsets(res, voxel_size, dev):
    lin = torch.linspace(-0.5, 0.5, res)                      # render_helpers.py:109-117
    xx, yy, zz = torch.meshgrid(lin, lin, lin, indexing="ij")
    return (torch.stack([xx, yy, zz], dim=-1).float().to(dev) * voxel_size).reshape(1, -1, 3)


@torch.no_grad()
def scores_device(sdf_network, map_states, voxel_size, bits=8, nodes=None, chunk=65536):
    """SDF on the res^3 lattice of the given octree nodes (default: every node that owns embeddings, i.e. the SURFACE leaves)
    -> (f32[len(nodes), res^3] on the device, nodes i64).  Same arithmetic as get_scores_once (render_helpers.py:104-146): lattice
    point = centre + linspace(-0.5, 0.5, res) * voxel_size, trilinear gather, decoder forward.  No host synchronisation."""
    dev = torch.device("cuda")
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    res = int(bits)
    if nodes is None:
        nodes = (m.vox2row[:, 0] >= 0).nonzero().view(-1)
    offs = _lattice_offsets(res, voxel_size, dev)
    bufs = DecoderBuffers.of(sdf_network, dev)
    bufs.refresh_transposes()
    out = torch.empty((nodes.shape[0], res ** 3), dtype=torch.float32, device=dev)
    chunk = max(1, chunk // (res ** 3) * 8)                   # voxels per launch (~0.5 M lattice points)
    for i in range(0, nodes.shape[0], chunk):
        idx = nodes[i:i + chunk]
        xyz = (offs + m.centres[idx].unsqueeze(1)).reshape(-1, 3).contiguous()
        vox = idx.to(torch.int32)[:, None].expand(-1, res ** 3).reshape(-1).contiguous()
        M = xyz.shape[0]
        feats = torch.empty((M, 16), dtype=torch.float32, device=dev)
        _capi.check(_capi.lib().nl_gather_trilinear_fwd(M, None, _capi.ptr(xyz), _capi.ptr(vox), _capi.ptr(m.centres),
                                                        _capi.ptr(m.vox2row), _capi.ptr(m.emb), float(voxel_size), _capi.ptr(feats),
                                                        _capi.stream_ptr()), "nl_gather_trilinear_fwd")
        _capi.LAUNCHES += 1
        mlp_forward(bufs, M, None, feats, out[i:i + idx.shape[0]].view(-1))
    return out, nodes


@torch.no_grad()
def get_scores(sdf_network, map_states, voxel_size, bits=8):
    """render_helpers.py:97-153: SDF on a res^3 lattice inside every voxel -> f32[n,res,res,res,1] (CPU).
    Nodes without embeddings (interior nodes, FEATURE-only leaves: vox2row = -1) gather an all-zero feature vector, so their whole
    lattice is the single value decoder(0) (the reference evaluates all res^3 points of each of them to get that constant): it is
    evaluated once and broadcast.  One device -> host copy at the end instead of one blocking .cpu() per 10 k-voxel chunk."""
    dev = torch.device("cuda")
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    res = int(bits)
    lat, nodes = scores_device(sdf_network, m, voxel_size, res)
    bufs = DecoderBuffers.of(sdf_network, dev)
    bufs.refresh_transposes()
    zero = torch.zeros((1, 16), dtype=torch.float32, device=dev)
    const = torch.empty(1, dtype=torch.float32, device=dev)
    mlp_forward(bufs, 1, None, zero, const)
    full = const.expand(m.n_nodes, res ** 3).clone()
    full[nodes] = lat
    return full.cpu().view(-1, res, res, res, 1)


# ======================================================================================================
# optimisation loops
# ======================================================================================================
def _seed_from_cuda(dev):
    """A fresh 32-bit seed drawn from torch's CUDA generator without a host round trip being needed later: a 1-element device tensor."""
    return torch.randint(1, 2 ** 31 - 1, (1,), device=dev, dtype=torch.int32)


def select_rays_device(dirs_all, gt_all, cos_all, n_select, n_dev=None, seed=None, out=None):
    """nl_select_rays: n_select distinct rays per scan, uniformly at random, in point order (the distribution of
    LidarFrame.sample_rays), gathered in the same launch.  dirs_all f32[F,cap,3] or [cap,3]; n_dev int64[F] device (None: all cap rows
    are points); seed int32[1] device tensor.  Returns (dirs [F*n_select,3], gt, cos)."""
    if dirs_all.dim() == 2:
        dirs_all, gt_all, cos_all = dirs_all[None], gt_all[None], cos_all[None]
    F, cap = dirs_all.shape[0], dirs_all.shape[1]
    dev = dirs_all.device
    if n_dev is None:
        n_dev = torch.full((F,), cap, dtype=torch.int64, device=dev)
    if out is None:
        out = (torch.empty((F * n_select, 3), dtype=torch.float32, device=dev), torch.empty(F * n_select, dtype=torch.float32, device=dev),
               torch.empty(F * n_select, dtype=torch.float32, device=dev))
    _capi.check(_capi.lib().nl_select_rays(F, cap, int(n_select), _capi.ptr(n_dev.view(-1)), _capi.ptr(seed), 0, _capi.ptr(dirs_all.contiguous()),
                                           _capi.ptr(gt_all.contiguous()), _capi.ptr(cos_all.contiguous()), _capi.ptr(out[0]), _capi.ptr(out[1]),
                                           _capi.ptr(out[2]), None, _capi.stream_ptr()), "nl_select_rays")
    _capi.LAUNCHES += 1
    return out


class _few_threads:
    """The reference's host-side ray selection is a handful of small element-wise CPU ops + a top-k over ~10^5 values; on a
    many-core host torch fans each of them out over every core and the fork/join costs far more than the work (measured on the
    128-CPU B200 box: 11 ms per frame and iteration, vs ~2 ms with 8 threads).  Same arithmetic, same RNG stream."""

    def __init__(self, n=8):
        self.n = n

    def __enter__(self):
        self.prev = torch.get_num_threads()
        if self.prev > self.n:
            torch.set_num_threads(self.n)

    def __exit__(self, *a):
        if torch.get_num_threads() != self.prev:
            torch.set_num_threads(self.prev)


_FRAME_ARRAYS = weakref.WeakKeyDictionary()


def _frame_arrays(f, dev):
    """Device copies of a scan's per-point data: unit directions f32[n,3], incidence cosines f32[n], cosine-corrected ranges f32[n]
    (criterion.py:30-32).  Computed once per frame OBJECT and kept in a weak-key side table: a keyframe stays in the optimisation
    window for many calls (window_size 4-8) and the tracked frame goes straight into the next mapping call, while re-uploading
    5 x 1.3 MB from pageable memory was ~10 % of a captured mapping call.  Tied to the identity of the frame's tensors (a frame whose
    points / cosines / directions are REPLACED is uploaded again); nothing is attached to the frame itself, so pickling a frame
    (the reference passes frames between its processes through queues) does not drag device memory along."""
    dev = torch.device(dev)
    src = (f.rays_d, f.pointsCos, f.points)
    try:
        c = _FRAME_ARRAYS.get(f)
    except TypeError:          # an unhashable / non-weakrefable frame type: no caching
        c = False
    if c and c[0] is src[0] and c[1] is src[1] and c[2] is src[2] and c[3].device.type == dev.type and \
            (dev.index is None or dev.index == c[3].device.index):
        return c[3], c[4], c[5]
    dirs = src[0].reshape(-1, 3).float().to(dev).contiguous()
    cos = src[1].float().view(-1).to(dev).contiguous()
    gt = torch.norm(src[2].float().to(dev), 2, -1) * cos
    if gt.is_cuda:
        # the arrays outlive this call and may next be read on another stream (tracker and mapper run on different ones): make
        # them complete now -- once per frame, and the uploads from pageable memory have stalled the host anyway
        torch.cuda.current_stream(gt.device).synchronize()
    if c is not False:
        try:
            _FRAME_ARRAYS[f] = src + (dirs, cos, gt)
        except TypeError:
            pass
    return dirs, cos, gt


class _FrameBatch:
    """Device copies of the per-frame point data (uploaded once per frame object instead of per iteration / per call)."""

    def __init__(self, frames, dev):
        self.frames = frames
        arrays = [_frame_arrays(f, dev) for f in frames]
        self.dirs = [a[0] for a in arrays]
        self.cos = [a[1] for a in arrays]
        self.gt = [a[2] for a in arrays]

    def select(self, N_rays, dev, track=False, mode="host"):
        """mode "host": ray selection like the reference (frame.sample_rays -> boolean mask, CPU torch RNG: the same seed
        picks the same rays as the reference), gathered on the device.  mode "device": the same distribution (uniform
        without replacement = top-k of iid keys, sample_util.py:4-19 with a constant mask) drawn with the CUDA generator,
        no host round trip; frame.sample_mask is not updated."""
        d, g, c, fid = [], [], [], []
        for i, f in enumerate(self.frames):
            if mode == "device":
                n = self.dirs[i].shape[0]
                k = min(N_rays, n)
                di, gi, ci = select_rays_device(self.dirs[i], self.gt[i], self.cos[i], k, n_dev=None, seed=_seed_from_cuda(dev))
                d.append(di); g.append(gi); c.append(ci)
                fid.append(torch.full((k,), i, dtype=torch.int32, device=dev))
                continue
            with _few_threads():
                f.sample_rays(N_rays, track=True) if track else f.sample_rays(N_rays)
                idx = f.sample_mask.view(-1).nonzero().view(-1).to(dev, non_blocking=True)
            d.append(self.dirs[i][idx]); g.append(self.gt[i][idx]); c.append(self.cos[i][idx])
            fid.append(torch.full((idx.shape[0],), i, dtype=torch.int32, device=dev))
        return torch.cat(d).contiguous(), torch.cat(g).contiguous(), torch.cat(c).contiguous(), torch.cat(fid).contiguous()


def _check_ctl(ctl, what):
    """Kernel error bits accumulated over a whole call (include/nerfloam_b200.h section 8).  Bit 2 (traversal stack) cannot be
    repaired by retrying; bit 1 (sample capacity) is handled by the callers (restore + redo with a larger engine)."""
    if ctl[_capi.CTL_ERROR] & 4:
        raise _capi.NerfLoamError(f"{what}: octree traversal stack overflow (octree deeper than the 18 levels of octree.cpp:39?)")


def _grown_capacity(cap, ctl):
    return max(2 * cap, int(ctl[_capi.CTL_MAX_SAMPLES] * 1.25) + 1024)


class _MapGraph:
    """One captured mapping iteration (per-frame ray selection -> rays -> traversal -> sampling -> gather -> decoder fwd/bwd ->
    embedding scatter / pose gradients -> Adam on embeddings, decoder and poses) with every per-call input in static device
    buffers.  At the reference's real iteration size (5 x 2048 rays, ~10^5 samples) an iteration is ~40 kernel launches of a
    few microseconds each: issued one by one from Python it is host-bound (1.3 ms), replayed as a graph it is not.
    Captured once per (map version, table, decoder, window shape); every call is num_iterations replays + ONE read-back."""

    _cache = {}

    def __init__(self, key, m, emb, sdf_network, cfg, F, N_rays, lrs, update_decoder, pose_rows, deterministic, cap, spr):
        dev = emb.device
        R = F * N_rays
        eng = SDFEngine(R, R * spr, dev)            # private: captured pointers must stay valid
        bufs = DecoderBuffers(sdf_network, dev)
        mg = MapState.__new__(MapState)              # the map as the graph sees it: same arrays, the table at the size that is optimised
        mg.__dict__.update(m.__dict__)
        mg.emb = emb
        m = mg
        self.key, self.eng, self.bufs, self.m, self.emb, self.F, self.N, self.cap = key, eng, bufs, m, emb, F, N_rays, cap
        self.packed = m.packed_children()
        self.dirs = torch.tensor([0.0, 0.0, -1.0], device=dev).repeat(F, cap, 1).contiguous()
        self.gt = torch.ones((F, cap), device=dev)
        self.cos = torch.ones((F, cap), device=dev)
        self.n_dev = torch.full((F, 1), cap, dtype=torch.int64, device=dev)
        self.sel_seed = torch.ones(1, dtype=torch.int32, device=dev)        # ray-selection stream, advanced inside the graph
        self.sel_out = (torch.empty((R, 3), device=dev), torch.empty(R, device=dev), torch.empty(R, device=dev))
        self.fid = torch.arange(F, dtype=torch.int32, device=dev).repeat_interleave(N_rays).contiguous()
        self.pose6 = torch.zeros((F, 6), device=dev)
        self.pose_m, self.pose_v = torch.zeros((F, 6), device=dev), torch.zeros((F, 6), device=dev)     # Adam moments of the poses (nl_pose_step)
        self.seed_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        any_pose = len(pose_rows) > 0
        groups = [dict(param=emb, grad=None, lr=lrs[0])]
        if update_decoder:
            groups += [dict(param=p.data, grad=g, lr=lrs[1]) for p, g in zip(bufs.params, bufs.grads)]
        state = {"opt": None}

        def body():
            # per frame: uniform without replacement among the scan's points, in point order, gathered -- one launch (csrc/select.cu)
            dirs, gt, cos = select_rays_device(self.dirs, self.gt, self.cos, N_rays, n_dev=self.n_dev, seed=self.sel_seed, out=self.sel_out)
            eng.rays_from_poses(self.pose6, dirs, self.fid)
            fused_tail = any_pose and F <= 31     # pose gradients + every pose's Adam step + loss read-out + both seed advances: one launch
            eng.forward_backward(m, bufs, R, cfg, gt, cos, dir_local=dirs, ray_frame=self.fid, n_frames=F, update_decoder=update_decoder,
                                 update_emb=True, update_pose=any_pose, pose6=self.pose6,
                                 rng_seed_dev=None if deterministic else self.seed_dev,
                                 pose_step=dict(mask=sum(1 << i for i in pose_rows), m=self.pose_m, v=self.pose_v, lr=lrs[2],
                                                seeds=[(self.sel_seed, 0x632BE5), (self.seed_dev, 0x3779B1)]) if fused_tail else None)
            if state["opt"] is None:
                groups[0]["grad"] = eng.grad_emb
                pg = [] if fused_tail else [dict(param=self.pose6[i], grad=eng.pose_grad[i], lr=lrs[2]) for i in pose_rows]
                state["opt"] = FusedAdam(groups + pg, ctl=eng.ctl)     # one fixed control block: forward_backward folds in place
            state["opt"].step()
            if not fused_tail:
                self.sel_seed.add_(0x632BE5)
                self.seed_dev.add_(0x3779B1)

        # one throw-away eager iteration on a side stream (allocations, one-time kernel attributes), then the capture; the
        # parameters it touches are put back afterwards
        keep = (emb.clone(), [p.data.clone() for p in bufs.params])
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            eng.begin_call()
            body()
        torch.cuda.current_stream(dev).wait_stream(side)
        l0 = _capi.LAUNCHES
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            body()
        self.launches_per_iter = _capi.LAUNCHES - l0 + 1
        self.opt = state["opt"]
        with torch.no_grad():
            emb.copy_(keep[0])
            for p, q in zip(bufs.params, keep[1]):
                p.data.copy_(q)

    @classmethod
    def get(cls, m, emb, sdf_network, cfg, F, N_rays, lrs, update_decoder, pose_rows, deterministic, n_points, spr):
        cap = max(1 << 17, 1 << (int(n_points) - 1).bit_length())
        stable = getattr(m, "stable", False)
        if stable and getattr(m, "emb_full", None) is not None and emb.data_ptr() == m.emb_full.data_ptr():
            # a mapping.MapUpdater map: every array sits in a capacity-sized buffer at a fixed address, so the captured graph stays
            # valid across map updates; the table is optimised at its full capacity (rows not yet handed out are zero, receive zero
            # gradients and therefore do not move under Adam)
            emb = m.emb_full
        key = (F, N_rays, tuple(float(x) for x in lrs), bool(update_decoder), tuple(pose_rows), bool(deterministic), cap, int(spr),
               m.centres.data_ptr(), m.structure.data_ptr(), m.vox2row.data_ptr(), m.packed_children().data_ptr(), emb.data_ptr(),
               -1 if stable else m.n_nodes, int(emb.shape[0]), tuple(p.data_ptr() for p in _decoder_params(sdf_network)),
               tuple(sorted(cfg.items())))
        g = cls._cache.get("g")
        if g is None or g.key != key:
            cls._cache = {}
            g = cls(key, m, emb, sdf_network, cfg, F, N_rays, lrs, update_decoder, pose_rows, deterministic, cap, spr)
            cls._cache = {"g": g}
        return g

    def _upload(self, frames):
        """The scans of this call into the graph's static buffers (device-to-device for frames seen before: _frame_arrays)."""
        for i, f in enumerate(frames):
            d, c, g = _frame_arrays(f, self.dirs.device)
            n = d.shape[0]
            self.dirs[i, :n].copy_(d)
            self.cos[i, :n].copy_(c)
            self.gt[i, :n].copy_(g)
            self.n_dev[i].fill_(n)

    def run(self, frames, pose6_init, num_iterations, seed):
        dev = self.dirs.device
        self._upload(frames)
        self.pose6.copy_(pose6_init)
        self.seed_dev.fill_(seed if seed < 2 ** 31 else seed - 2 ** 32)
        self.sel_seed.copy_(_seed_from_cuda(dev))          # ray selection follows torch's CUDA generator (torch.manual_seed reproduces it)
        for g in self.opt.groups:
            g["m"].zero_(); g["v"].zero_()
        self.pose_m.zero_(); self.pose_v.zero_()
        self.eng.begin_call()
        for _ in range(num_iterations):
            self.graph.replay()
        _capi.LAUNCHES += self.launches_per_iter * num_iterations
        return self.eng.read_ctl()


def bundle_adjust_frames(keyframe_graph, embeddings, map_states, sdf_network, loss_criteria, voxel_size, step_size,
                         N_rays=512, num_iterations=10, truncation=0.1, max_voxel_hit=10, max_distance=10,
                         learning_rate=[1e-2, 1e-2, 5e-3], update_pose=True, update_decoder=True, profiler=None,
                         deterministic=False, noise_per_iter=None, loss_log=None, ray_selection="device", cuda_graph=None):
    """render_helpers.py:321-425.  Mutates `embeddings` (bf16 CUDA table), the decoder parameters and the
    frame poses in place, like the reference.  Returns None.  ray_selection: see _FrameBatch.select ("device" by default;
    "host" reproduces the reference's CPU RNG stream ray for ray).  cuda_graph (default: on whenever ray_selection="device" and no
    per-iteration host inputs/outputs are requested): the iteration is captured once per map version and replayed (_MapGraph).

    No host synchronisation per iteration: kernel error bits, "nothing was hit" iterations (which the reference skips,
    :405-409) and Adam's step count are tracked in a device-side control block that the Adam kernels read; the host looks at it
    once at the end of the call.  If the sample capacity was exceeded in any iteration the parameters and the RNG state are
    restored and the whole call is redone with a larger engine, so a truncated sample set never reaches the parameters."""
    if ray_selection not in ("host", "device"):
        raise ValueError("ray_selection must be 'host' or 'device'")
    dev = embeddings.device
    if dev.type != "cuda":
        raise RuntimeError("bundle_adjust_frames runs on the GPU only (no CPU fallback)")
    frames = list(keyframe_graph)
    F = len(frames)
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    emb = embeddings.detach()
    if not (emb.dtype == torch.bfloat16 and emb.is_contiguous()):
        raise RuntimeError("embeddings must be a contiguous bf16 CUDA tensor (mapping.py:305-314)")
    m.emb = emb
    cfg = _cfg(step_size, voxel_size, max_distance, loss_criteria)
    bufs = DecoderBuffers(sdf_network, dev)
    R = N_rays * F
    batch = _FrameBatch(frames, dev)
    pose6 = torch.stack([f.pose.data.detach().float().cpu() for f in frames]).to(dev).contiguous()
    pose_opt = [(f.index != 0 and update_pose) for f in frames]   # render_helpers.py:346-351
    for f, po in zip(frames, pose_opt):
        if po:
            f.pose.requires_grad_(True)
    # decoder weight gradients + the decoder's Adam stay on the engine's side stream and are joined right before the next
    # iteration's decoder (engine.SDFEngine.forward_backward, defer_wgrad): same arithmetic, shorter critical path
    pipeline = update_decoder and os.environ.get("NL_PIPELINE", "1") != "0"
    pose_rows = [i for i, po in enumerate(pose_opt) if po]
    pose_params = [pose6[i] for i in pose_rows]                    # views into pose6 (contiguous rows)

    def run(eng):
        eng.begin_call()
        groups = [dict(param=emb, grad=None, lr=learning_rate[0])]
        if update_decoder:
            groups += [dict(param=p.data, grad=g, lr=learning_rate[1], side=True) for p, g in zip(bufs.params, bufs.grads)]
        opt = None
        for it in range(num_iterations):
            dirs, gt, cos, fid = batch.select(N_rays, dev, mode=ray_selection)
            eng.rays_from_poses(pose6, dirs, fid)
            noise = noise_per_iter[it] if noise_per_iter is not None else None
            seed = 0 if (deterministic or noise is not None) else _seed_from_torch()
            eng.forward_backward(m, bufs, dirs.shape[0], cfg, gt, cos, dir_local=dirs, ray_frame=fid, n_frames=F, noise=noise,
                                 rng_seed=seed, update_decoder=update_decoder, update_emb=True, update_pose=any(pose_opt), pose6=pose6,
                                 defer_wgrad=pipeline)
            if opt is None:
                groups[0]["grad"] = eng.grad_emb
                pg = [dict(param=pose_params[k], grad=eng.pose_grad[i], lr=learning_rate[2]) for k, i in enumerate(pose_rows)]
                opt = FusedAdam(groups + pg, ctl=lambda: eng.ctl)
            if loss_log is not None:                    # diagnostic path: one read-back per iteration
                st = eng.read_stats()
                if not (st.n_hit_rays <= 0 or (st.error & 1)):
                    loss_log.append(st.loss)
            opt.step(side_stream=eng.deferred_stream())
        eng.join_side()
        return eng.read_ctl()

    graph_ok = ray_selection == "device" and noise_per_iter is None and loss_log is None and \
        all(f.points.shape[0] >= N_rays for f in frames)
    if cuda_graph is None:
        # automatic only for maps whose arrays keep their addresses across map updates (mapping.MapUpdater): a capture costs about
        # as much as 1.5 eager calls, so re-capturing for every new map (the reference's per-frame dicts) would be a net loss
        cuda_graph = graph_ok and getattr(m, "stable", False)
    elif cuda_graph and not graph_ok:
        raise ValueError("cuda_graph=True needs ray_selection='device', no per-iteration host inputs/outputs and >= N_rays points per scan")
    cap = R * SAMPLES_PER_RAY_MAP
    while True:
        snap = (emb.clone(), [p.data.clone() for p in bufs.params] if update_decoder else None, pose6.clone(),
                torch.get_rng_state(), torch.cuda.get_rng_state(dev))
        n_log = len(loss_log) if loss_log is not None else 0
        if cuda_graph:
            g = _MapGraph.get(m, emb, sdf_network, cfg, F, N_rays, learning_rate, update_decoder, pose_rows, deterministic,
                              max(f.points.shape[0] for f in frames), -(-cap // R))
            ctl = g.run(frames, pose6, num_iterations, 0 if deterministic else _seed_from_torch())
            pose6.copy_(g.pose6)
        else:
            eng = _engine(R, cap, dev)
            ctl = run(eng)
        _check_ctl(ctl, "bundle_adjust_frames")
        if not (ctl[_capi.CTL_ERROR] & 2):
            break
        # sample capacity exceeded somewhere in the call: undo it and redo it with room for the largest iteration seen
        with torch.no_grad():
            emb.copy_(snap[0]); pose6.copy_(snap[2])
            if snap[1] is not None:
                for p, q in zip(bufs.params, snap[1]):
                    p.data.copy_(q)
        torch.set_rng_state(snap[3]); torch.cuda.set_rng_state(snap[4], dev)
        if loss_log is not None:
            del loss_log[n_log:]
        cap = _grown_capacity(cap, ctl)
    for _ in range(ctl[_capi.CTL_SKIPPED]):
        print("Encouter a bug while Mapping, currently not be fixed, Continue!!")  # render_helpers.py:407-409 (the step was skipped)
    with torch.no_grad():
        host = pose6.cpu()
        for i, f in enumerate(frames):
            if pose_opt[i]:
                f.pose.data.copy_(host[i].to(f.pose.data.device))


class _TrackGraph:
    """One captured tracking iteration (ray selection -> rays -> traversal -> sampling -> gather -> decoder fwd/bwd -> pose gradient
    -> Adam) with every per-scan input in static device buffers, so that the capture (tens of ms) is paid once per map / decoder
    version and every scan is 25 graph replays plus one statistics read-back."""

    _cache = {}
    _max_live = 4

    def __init__(self, key, m, sdf_network, cfg, N_rays, lr, deterministic, cap, samples_per_ray=64):
        dev = m.centres.device
        # a private engine: the shared ones may re-allocate buffers (pose accumulators, scratch) between scans, which would leave
        # the captured graph with dangling pointers
        eng = SDFEngine(N_rays, N_rays * samples_per_ray, dev)
        bufs = DecoderBuffers(sdf_network, dev)
        self.key, self.eng, self.cap, self.N = key, eng, cap, N_rays
        self.m, self.bufs, self.packed = m, bufs, m.packed_children()   # keep the captured tensors alive
        self.dirs = torch.tensor([0.0, 0.0, -1.0], device=dev).repeat(cap, 1)   # valid unit rays for the throw-away warm-up iteration
        self.gt = torch.ones(cap, device=dev)
        self.cos = torch.ones(cap, device=dev)
        self.n_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.pose6 = torch.zeros((1, 6), device=dev)
        self.seed_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.sel_seed = torch.ones(1, dtype=torch.int32, device=dev)        # ray-selection stream, advanced inside the graph
        self.sel_out = (torch.empty((N_rays, 3), device=dev), torch.empty(N_rays, device=dev), torch.empty(N_rays, device=dev))
        self.adam_m, self.adam_v = torch.zeros(6, device=dev), torch.zeros(6, device=dev)
        lib = _capi.lib()

        def body():
            # uniform without replacement among the scan's n points, in point order, gathered -- one launch (csrc/select.cu)
            dirs, gt, cos = select_rays_device(self.dirs, self.gt, self.cos, N_rays, n_dev=self.n_dev, seed=self.sel_seed, out=self.sel_out)
            eng.rays_from_poses(self.pose6, dirs, None)
            # Adam's step count, the "nothing hit" skip and the sticky error bits live in the engine's control block (one fixed
            # block: forward_backward folds this iteration's statistics into it in place); the iteration ends with ONE launch for
            # pose gradient + the pose's Adam step + loss read-out + the advance of the two RNG seeds (nl_pose_step)
            eng.forward_backward(m, bufs, N_rays, cfg, gt, cos, dir_local=dirs, ray_frame=None, n_frames=1, update_decoder=False,
                                 update_emb=False, update_pose=True, pose6=self.pose6, refresh_weights=False,
                                 rng_seed_dev=None if deterministic else self.seed_dev,
                                 pose_step=dict(mask=1, m=self.adam_m, v=self.adam_v, lr=lr, seeds=[(self.sel_seed, 0x632BE5), (self.seed_dev, 0x3779B1)]))

        # one throw-away eager iteration on a side stream (allocations, one-time kernel attributes), then the capture
        bufs.refresh_transposes()
        self.n_dev.fill_(cap)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            body()
        torch.cuda.current_stream(dev).wait_stream(side)
        l0 = _capi.LAUNCHES
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            body()
        self.launches_per_iter = _capi.LAUNCHES - l0 + 1

    @classmethod
    def get(cls, m, sdf_network, cfg, N_rays, lr, deterministic, n_points, samples_per_ray=64):
        cap = max(1 << 17, 1 << (int(n_points) - 1).bit_length())
        stable = getattr(m, "stable", False)      # mapping.MapUpdater map: fixed base addresses, the graph survives map updates
        key = (N_rays, float(lr), bool(deterministic), cap, int(samples_per_ray), m.centres.data_ptr(), m.structure.data_ptr(), m.vox2row.data_ptr(),
               m.packed_children().data_ptr(), m.emb.data_ptr(), -1 if stable else m.n_nodes, -1 if stable else int(m.emb.shape[0]),
               tuple(p.data_ptr() for p in _decoder_params(sdf_network)), tuple(sorted(cfg.items())))
        g = cls._cache.pop(key, None)
        if g is None:
            # a few live graphs, least recently used first out: the tracker of a running system alternates between the two snapshot
            # slots of share.SharedMap (two tables, two decoder copies) and uses a different rate for the first scans
            if not stable:
                cls._cache.clear()                              # a per-frame map (reference dict): its arrays die with it, keep nothing else alive
            while len(cls._cache) >= cls._max_live:
                cls._cache.pop(next(iter(cls._cache)))
            g = cls(key, m, sdf_network, cfg, N_rays, lr, deterministic, cap, samples_per_ray)
        cls._cache[key] = g                                     # (re-)inserted last = most recently used
        return g

    def _upload(self, frame):
        """The scan into the graph's static buffers; its device arrays stay cached for the mapping call that follows (_frame_arrays)."""
        d, c, g = _frame_arrays(frame, self.dirs.device)
        n = d.shape[0]
        self.dirs[:n].copy_(d)
        self.cos[:n].copy_(c)
        self.gt[:n].copy_(g)
        self.n_dev.fill_(n)

    def run(self, frame, pose6_init, num_iterations, seed):
        dev = self.dirs.device
        self.bufs.refresh_transposes()        # the decoder may have been updated in place since the capture (same pointers, new values)
        self._upload(frame)
        self.pose6.copy_(pose6_init)
        self.seed_dev.fill_(seed if seed < 2 ** 31 else seed - 2 ** 32)
        self.sel_seed.copy_(_seed_from_cuda(dev))          # ray selection follows torch's CUDA generator (torch.manual_seed reproduces it)
        self.adam_m.zero_(); self.adam_v.zero_()
        self.eng.begin_call()
        for _ in range(num_iterations):
            self.graph.replay()
        _capi.LAUNCHES += self.launches_per_iter * num_iterations
        return self.eng.read_stats(), self.eng.read_ctl()


def _track_frame_graph(frame_pose, curr_frame, map_states, sdf_network, loss_criteria, voxel_size, N_rays, step_size, num_iterations,
                       learning_rate, max_distance, deterministic):
    dev = torch.device("cuda")
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    cfg = _cfg(step_size, voxel_size, max_distance, loss_criteria)
    init_pose = deepcopy(frame_pose).cuda()
    init_pose.requires_grad_(True)
    lr = learning_rate * 2 if curr_frame.index < 2 else learning_rate / 3   # render_helpers.py:448-450
    n_points = curr_frame.points.shape[0]
    if n_points < N_rays:
        raise ValueError("cuda_graph=True needs at least N_rays points in the scan")
    seed = 0 if deterministic else _seed_from_torch()
    spr = SAMPLES_PER_RAY_TRACK
    while True:
        g = _TrackGraph.get(m, sdf_network, cfg, N_rays, lr, deterministic, n_points, spr)
        eng = g.eng
        st, ctl = g.run(curr_frame, init_pose.data.detach().reshape(1, 6), num_iterations, seed)
        _check_ctl(ctl, "track_frame")
        if not (ctl[_capi.CTL_ERROR] & 2):
            break
        spr = -(-_grown_capacity(N_rays * spr, ctl) // N_rays)       # sample capacity exceeded: re-capture with a larger engine, redo the scan
    with torch.no_grad():
        init_pose.data.copy_(g.pose6.reshape(init_pose.data.shape))
    if ctl[_capi.CTL_SKIPPED] > 0 or st.n_samples == 0:
        print("Encouter a bug while Tracking, currently not be fixed, Restarting!!")  # render_helpers.py:488-491
        return init_pose, None
    return init_pose, (eng.hit_rank[:N_rays] >= 0).clone()


def track_frame(frame_pose, curr_frame, map_states, sdf_network, loss_criteria, voxel_size, N_rays=512, step_size=0.05,
                num_iterations=10, truncation=0.1, learning_rate=1e-3, max_voxel_hit=10, max_distance=10, profiler=None,
                depth_variance=False, deterministic=False, noise_per_iter=None, loss_log=None, ray_selection="device",
                cuda_graph=None):
    """render_helpers.py:428-514: optimise the 6-vector pose of one scan against a frozen map.
    Returns (OptimizablePose on the GPU, hit_mask bool[N_rays]) or (pose, None) if nothing was hit.
    ray_selection: see _FrameBatch.select.  cuda_graph=True (needs ray_selection="device"): the iteration -- ray selection,
    rays, traversal, sampling, gather, decoder forward/backward, pose gradient, Adam -- is captured once and replayed, with
    the sampler seed and the Adam step count in device memory; the host looks at the statistics once at the end instead of
    every iteration (an iteration without hits makes the call return (pose, None) like the reference, just later)."""
    if ray_selection not in ("host", "device"):
        raise ValueError("ray_selection must be 'host' or 'device'")
    graph_ok = ray_selection == "device" and noise_per_iter is None and loss_log is None and curr_frame.points.shape[0] >= N_rays
    if cuda_graph is None:          # default: the captured path for maps with stable addresses (mapping.MapUpdater), see bundle_adjust_frames
        stable = getattr(map_states, "stable", False) or getattr(map_states.get("_mapstate") if isinstance(map_states, dict) else None, "stable", False)
        cuda_graph = graph_ok and stable
    if cuda_graph:
        if not graph_ok:
            raise ValueError("cuda_graph=True needs ray_selection='device', no per-iteration host inputs/outputs and >= N_rays points")
        return _track_frame_graph(frame_pose, curr_frame, map_states, sdf_network, loss_criteria, voxel_size, N_rays, step_size,
                                  num_iterations, learning_rate, max_distance, deterministic)
    dev = torch.device("cuda")
    m = map_states if isinstance(map_states, MapState) else MapState.from_map_states(map_states, dev)
    cfg = _cfg(step_size, voxel_size, max_distance, loss_criteria)
    bufs = DecoderBuffers(sdf_network, dev)
    init_pose = deepcopy(frame_pose).cuda()
    init_pose.requires_grad_(True)
    pose6 = init_pose.data.detach().reshape(1, 6).contiguous()     # shares storage with the parameter
    lr = learning_rate * 2 if curr_frame.index < 2 else learning_rate / 3   # render_helpers.py:448-450
    cap = N_rays * SAMPLES_PER_RAY_TRACK
    eng = _engine(N_rays, cap, dev)
    eng.begin_call()
    batch = _FrameBatch([curr_frame], dev)
    opt = None
    hit_mask = None
    n_last = 0
    bufs.refresh_transposes()           # the decoder is frozen while tracking: derive the kernel-side weight images once
    for it in range(num_iterations):
        dirs, gt, cos, fid = batch.select(N_rays, dev, track=True, mode=ray_selection)
        noise = noise_per_iter[it] if noise_per_iter is not None else None
        seed = 0 if (deterministic or noise is not None) else _seed_from_torch()
        while True:
            eng.rays_from_poses(pose6, dirs, None)
            eng.forward_backward(m, bufs, dirs.shape[0], cfg, gt, cos, dir_local=dirs, ray_frame=None, n_frames=1, noise=noise,
                                 rng_seed=seed, update_decoder=False, update_emb=False, update_pose=True, pose6=pose6,
                                 refresh_weights=False)
            st = eng.read_stats()   # the reference syncs here too (hit_mask, None checks)
            if st.error & 4:
                _check_ctl([4], "track_frame")
            if not (st.error & 2):
                break
            # sample capacity exceeded: nothing has been applied yet (the optimiser step follows) -- redo this iteration on a larger engine
            cap = max(2 * cap, int(st.n_samples * 1.25) + 1024)
            eng = _engine(N_rays, cap, dev)
            if opt is not None:
                opt.groups[0]["grad"] = None
        if st.n_hit_rays <= 0 or (st.error & 1) or st.n_samples == 0:
            print("Encouter a bug while Tracking, currently not be fixed, Restarting!!")  # render_helpers.py:488-491
            n_last = 0
            break
        n_last = dirs.shape[0]
        if loss_log is not None:
            loss_log.append(st.loss)
        if opt is None:
            opt = FusedAdam([dict(param=pose6[0], grad=eng.pose_grad[0], lr=lr)])
        opt.groups[0]["grad"] = eng.pose_grad[0]
        opt.step()
    if n_last:
        hit_mask = (eng.hit_rank[:n_last] >= 0).clone()   # of the last iteration, like the reference's return value
    return init_pose, hit_mask
