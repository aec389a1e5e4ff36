"""SDFEngine: the fused per-iteration pipeline (rays -> samples -> features -> SDF -> loss -> gradients)
as a chain of C-ABI kernel launches on one CUDA stream, with persistent device buffers and no host
synchronisation inside an iteration.

This is the host-side orchestration of SURVEY.md section 8 a-2 .. a-12; the arithmetic is all in
libnerfloam_b200.so.  torch is used for device memory and streams only.
"""
import contextlib
import ctypes as C
import os

import torch

from . import _capi
from ._capi import MlpGrads, MlpWeights, RenderArgs, RenderStats

STATS_BYTES = C.sizeof(RenderStats)
N_SAMPLES_OFFSET = RenderStats.n_samples.offset


def mlp_impl(width):
    """'tc' = tcgen05 3xTF32 tensor-core kernels (width 256), 'simt' = fp32 CUDA-core kernels.  NL_MLP_IMPL overrides."""
    want = os.environ.get("NL_MLP_IMPL", "tc")
    return "tc" if (want == "tc" and width == 256) else "simt"


def mlp_forward(bufs, M_cap, M_dev, feats, sdf):
    """sdf[M] = decoder(feats[M,16]) through the selected kernel implementation."""
    lib, st = _capi.lib(), _capi.stream_ptr()
    if mlp_impl(bufs.width) == "tc":
        p = bufs.params
        _capi.check(lib.nl_mlp_tc_forward(M_cap, M_dev, _capi.ptr(feats), _capi.ptr(bufs.tc_panels), _capi.ptr(p[1]), _capi.ptr(p[3]),
                                          _capi.ptr(p[4]), _capi.ptr(p[5]), _capi.ptr(sdf), st), "nl_mlp_tc_forward")
    else:
        w = bufs.weights_struct()
        _capi.check(lib.nl_mlp_forward(M_cap, M_dev, _capi.ptr(feats), C.byref(w), _capi.ptr(sdf), st), "nl_mlp_forward")
    _capi.LAUNCHES += 1


def mlp_train(bufs, M_cap, M_dev, feats, sdf, dfeats, want_wgrad, act, s_flag=None, s_depth=None, s_ray=None, cos=None, gt_depth=None,
              stats_ptr=None, truncation=0.0, dsdf_ext=None, wgrad_stream=None):
    """Forward + (loss | external d sdf) + backward.  act: dict with scratch tensors for the weight gradients
    ('h1','dh2' [cap,W] for simt; one 'buf' of nl_mlp_tc_act_floats(cap) floats for tc).  Accumulates into bufs.grads when want_wgrad."""
    lib, st = _capi.lib(), _capi.stream_ptr()
    gs = bufs.grads_struct() if want_wgrad else None
    gp = C.byref(gs) if want_wgrad else None
    if mlp_impl(bufs.width) == "tc":
        p = bufs.params
        _capi.check(lib.nl_mlp_tc_train(M_cap, M_dev, _capi.ptr(feats), _capi.ptr(bufs.tc_panels), _capi.ptr(p[2]), _capi.ptr(p[1]), _capi.ptr(p[3]),
                                        _capi.ptr(p[4]), _capi.ptr(p[5]), _capi.ptr(s_flag), _capi.ptr(s_depth), _capi.ptr(s_ray),
                                        _capi.ptr(cos), _capi.ptr(gt_depth), stats_ptr, float(truncation), _capi.ptr(sdf),
                                        _capi.ptr(dfeats), gp, _capi.ptr(act["buf"]) if want_wgrad else None, _capi.ptr(dsdf_ext),
                                        C.c_void_p(wgrad_stream.cuda_stream) if (want_wgrad and wgrad_stream is not None) else None, st),
                    "nl_mlp_tc_train")
        _capi.LAUNCHES += 4 if want_wgrad else 1
    else:
        w = bufs.weights_struct()
        _capi.check(lib.nl_mlp_train(M_cap, M_dev, _capi.ptr(feats), C.byref(w), _capi.ptr(s_flag), _capi.ptr(s_depth), _capi.ptr(s_ray),
                                     _capi.ptr(cos), _capi.ptr(gt_depth), stats_ptr, float(truncation), _capi.ptr(sdf), _capi.ptr(dfeats),
                                     gp, _capi.ptr(act["h1"]) if want_wgrad else None, _capi.ptr(act["dh2"]) if want_wgrad else None,
                                     _capi.ptr(dsdf_ext), st), "nl_mlp_train")
        _capi.LAUNCHES += 2 if want_wgrad else 1


def alloc_act(width, M_cap, device):
    """Scratch for the decoder weight gradients, sized for M_cap samples."""
    if mlp_impl(width) == "tc":
        n = int(_capi.lib().nl_mlp_tc_act_floats(int(M_cap)))
        return {"buf": torch.empty(n, dtype=torch.float32, device=device)}
    return {k: torch.empty((int(M_cap), width), dtype=torch.float32, device=device) for k in ("h1", "dh2")}


def pack_children(centres, structure):
    """nl_octree_pack_children: [n, 8] records {child centre, child id} (128 B per node) for the cooperative traversal kernel.
    Checks the octree invariant it relies on (a child's side is half its parent's, octree.cpp:51-111)."""
    n = centres.shape[0]
    ch = structure[:, :8].long()
    present = ch >= 0
    child_side = structure[ch.clamp(min=0), 8]
    if not bool(((child_side * 2 == structure[:, 8:9]) | ~present).all()):
        raise _capi.NerfLoamError("octree structure violates side(child) == side(parent) / 2")
    packed = torch.empty(int(_capi.lib().nl_octree_packed_bytes(n)), dtype=torch.uint8, device=centres.device)
    _capi.check(_capi.lib().nl_octree_pack_children(n, _capi.ptr(centres), _capi.ptr(structure), _capi.ptr(packed), _capi.stream_ptr()),
                "nl_octree_pack_children")
    _capi.LAUNCHES += 1
    return packed


class MapState:
    """Device-resident map in hot-path layout: centres f32[n,3], structure i32[n,9], vox2row i32[n,8],
    emb bf16[V,16].  Built from the reference's map_states dict (mapping.py:328-337) by composing
    voxel_vertex_idx with voxel_id2embedding_id once per map update (instead of the 8 GB CPU lookup
    and the D2H/H2D detour of get_features, render_helpers.py:88, on every chunk of every iteration)."""

    def __init__(self, centres, structure, vox2row, emb, device="cuda"):
        self.centres = centres.detach().to(device=device, dtype=torch.float32).contiguous()
        self.structure = structure.detach().to(device=device, dtype=torch.int32).contiguous()
        self.vox2row = vox2row.detach().to(device=device, dtype=torch.int32).contiguous()
        self.emb = emb if (emb.is_cuda and emb.dtype == torch.bfloat16 and emb.is_contiguous()) else \
            emb.detach().to(device=device, dtype=torch.bfloat16).contiguous()
        assert self.centres.shape[1] == 3 and self.structure.shape[1] == 9 and self.vox2row.shape[1] == 8
        assert self.emb.shape[1] == 16, "embedding dim must be 16 (decoder_specs.in_dim of every shipped config)"
        self.n_nodes = self.centres.shape[0]
        self._packed = None

    _cache = {}

    def packed_children(self):
        """Traversal image of the octree (nl_octree_pack_children), built once per map version."""
        if getattr(self, "_packed", None) is None:
            self._packed = pack_children(self.centres, self.structure)
            if getattr(self, "_cache_ref", None) is not None:
                self._cache_ref["packed"] = self._packed
        return self._packed

    @staticmethod
    def _fingerprint(map_states):
        """Content fingerprint of the structural part of a reference map_states dict.  The dict is rebuilt (and, in the tracker
        process, freshly unpickled) for every frame, so tensor identity / _version say nothing: a freed tensor's address is
        readily reused and an update that only turns FEATURE leaves into SURFACE leaves keeps every shape.  CRC-32 of the three
        structural tensors costs ~25 ms per 10^6 nodes on the host (they are CPU tensors in the reference), against a full
        re-composition through the id table + upload + re-packing."""
        import zlib
        vidx = map_states["voxel_vertex_idx"].detach()
        n = int(vidx.shape[0])

        def h(t, dtype):
            a = t.detach().to(device="cpu", dtype=dtype).contiguous().numpy()
            return zlib.crc32(memoryview(a).cast("B"))
        stru = map_states.get("voxel_structure")      # absent in the encoder_states dict of Mapping.extract_mesh (mapping.py:363-371)
        # the id table is hashed over the entries a vertex id can address (vertex ids are node ids < n; the reference allocates 2e9)
        id2 = map_states["voxel_id2embedding_id"].detach().reshape(-1)
        return (n, h(vidx, torch.int32), h(stru, torch.int32) if stru is not None else -1, h(map_states["voxel_center_xyz"], torch.float32),
                int(id2.shape[0]), h(id2[:max(n, int(vidx.max()) + 1 if vidx.numel() else 0)], torch.int32))

    @classmethod
    def from_map_states(cls, map_states, device="cuda"):
        """map_states: the reference dict (mapping.py:328-337).  A dict produced by mapping.MapUpdater carries the finished
        MapState ("_mapstate") and is used as is; for the reference's own dict the derived arrays (voxel -> row table, device
        copies, packed traversal image) are cached on a content fingerprint of its index tensors."""
        own = map_states.get("_mapstate")
        if isinstance(own, MapState) and own.centres.device == torch.device(device):
            return own
        key = cls._fingerprint(map_states)
        if cls._cache.get("key") != key:
            v = map_states["voxel_vertex_idx"].detach().cpu().long()
            flat = map_states["voxel_id2embedding_id"].detach().cpu().reshape(-1)
            rows = torch.where(v >= 0, flat[v.clamp(min=0)].long(), torch.full_like(v, -1))
            stru = map_states.get("voxel_structure")
            if stru is None:      # meshing-only dict (mapping.py:363-371): rows are SURFACE voxels, nothing is ever traversed
                stru = torch.cat([torch.full((v.shape[0], 8), -1, dtype=torch.int32), torch.ones((v.shape[0], 1), dtype=torch.int32)], 1)
            cls._cache = {"key": key, "vox2row": rows.to(torch.int32).to(device).contiguous(),
                          "centres": map_states["voxel_center_xyz"].detach().to(device=device, dtype=torch.float32).contiguous(),
                          "structure": stru.detach().to(device=device, dtype=torch.int32).contiguous(), "packed": None}
        c = cls._cache
        obj = cls.__new__(cls)
        obj.centres, obj.structure, obj.vox2row = c["centres"], c["structure"], c["vox2row"]
        obj._packed = c["packed"]
        obj._cache_ref = c                     # packed_children() stores the traversal image back into the shared cache entry
        emb = map_states["voxel_vertex_emb"]
        obj.emb = emb.detach() if (emb.is_cuda and emb.dtype == torch.bfloat16 and emb.is_contiguous()) else \
            emb.detach().to(device=device, dtype=torch.bfloat16).contiguous()
        obj.n_nodes = obj.centres.shape[0]
        return obj


class DecoderBuffers:
    """Flat device views of the decoder parameters for the kernels + transposes + fp32 gradient buffers.
    DecoderBuffers.of(decoder, device) returns a cached instance per decoder module (weakly referenced, validated against the
    parameters' addresses): the drop-in entry points are called once per scan / per autograd node, and re-allocating 1.6 MB of weight
    panels + gradient buffers each time is pure overhead.  The kernel-side weight images are still re-derived from the parameters
    whenever they are used (refresh_transposes): the optimiser kernels update parameters through raw pointers."""
    _cache = None

    @classmethod
    def of(cls, decoder, device):
        import weakref
        if cls._cache is None:
            cls._cache = weakref.WeakKeyDictionary()
        lin = list(decoder.pts_linears)
        key = (str(device), mlp_impl(lin[0].weight.shape[0])) + tuple(p.data_ptr() for p in (lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias,
                                                                                            decoder.sdf_out.weight, decoder.sdf_out.bias))
        hit = cls._cache.get(decoder)
        if hit is None or hit[0] != key:
            hit = (key, cls(decoder, device))
            cls._cache[decoder] = hit
        return hit[1]

    def __init__(self, decoder, device):
        lin = list(decoder.pts_linears)
        if len(lin) != 2 or getattr(decoder, "skips", []) not in ([], None):
            raise NotImplementedError("fused decoder kernel supports depth=2, skips=[] (every shipped config)")
        self.params = [lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, decoder.sdf_out.weight, decoder.sdf_out.bias]
        W = lin[0].weight.shape[0]
        if lin[0].weight.shape[1] != 16 or tuple(lin[1].weight.shape) != (W, W) or W not in (32, 64, 128, 256):
            raise NotImplementedError(f"unsupported decoder shape in_dim={lin[0].weight.shape[1]} width={W}")
        for p in self.params:
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
                raise RuntimeError("decoder parameters must be contiguous fp32 CUDA tensors (call decoder.cuda())")
        self.width = W
        self.W0t = torch.empty((16, W), device=device, dtype=torch.float32)
        self.W1t = torch.empty((W, W), device=device, dtype=torch.float32)
        # fp32 gradient accumulators as views into ONE flat buffer: a single zero-fill and, multi-GPU, a single all-reduce per iteration
        offs, n = [], 0
        for p in self.params:
            offs.append(n)
            n += (p.numel() + 63) // 64 * 64
        self.gradflat = torch.zeros(n, dtype=torch.float32, device=device)
        self.grads = [self.gradflat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, self.params)]
        self.tc_panels = None
        if mlp_impl(W) == "tc":
            self.tc_panels = torch.empty(int(_capi.lib().nl_mlp_tc_panel_bytes()), dtype=torch.uint8, device=device)

    def weights_struct(self):
        p = self.params
        return MlpWeights(self.width, *[C.c_void_p(t.data_ptr()) for t in p], C.c_void_p(self.W0t.data_ptr()),
                          C.c_void_p(self.W1t.data_ptr()))

    def grads_struct(self):
        return MlpGrads(*[C.c_void_p(g.data_ptr()) for g in self.grads])

    def refresh_transposes(self):
        """Re-derive the kernel-side weight images from the parameters (they change every optimiser step)."""
        if self.tc_panels is not None:
            _capi.check(_capi.lib().nl_mlp_tc_prepare(_capi.ptr(self.params[0]), _capi.ptr(self.params[2]), _capi.ptr(self.params[4]), _capi.ptr(self.tc_panels),
                                                      _capi.stream_ptr()), "nl_mlp_tc_prepare")
            _capi.LAUNCHES += 1
        else:
            _capi.check(_capi.lib().nl_mlp_prepare(self.width, _capi.ptr(self.params[0]), _capi.ptr(self.params[2]), _capi.ptr(self.W0t),
                                                   _capi.ptr(self.W1t), _capi.stream_ptr()), "nl_mlp_prepare")
            _capi.LAUNCHES += 2


class SDFEngine:
    """Persistent buffers for up to `max_rays` rays and `max_samples` samples per iteration."""

    def __init__(self, max_rays, max_samples, device="cuda", width=256, want_decoder_grads=True):
        self.device = torch.device(device)
        self.max_rays, self.max_samples = int(max_rays), int(max_samples)
        d = self.device
        R, M = self.max_rays, self.max_samples
        f32, i32 = torch.float32, torch.int32
        self.ws_bytes = int(_capi.lib().nl_render_workspace_bytes(R))
        self.workspace = torch.empty(self.ws_bytes, dtype=torch.uint8, device=d)
        self.stats = torch.zeros(STATS_BYTES, dtype=torch.uint8, device=d)
        self.ray_o = torch.empty((R, 3), dtype=f32, device=d)
        self.ray_d = torch.empty((R, 3), dtype=f32, device=d)
        self.hit_rank = torch.empty(R, dtype=i32, device=d)
        self.ray_nsamp = torch.empty(R, dtype=i32, device=d)
        self.ray_offset = torch.empty(R, dtype=i32, device=d)
        self.s_ray = torch.empty(M, dtype=i32, device=d)
        self.s_vox = torch.empty(M, dtype=i32, device=d)
        self.s_depth = torch.empty(M, dtype=f32, device=d)
        self.s_xyz = torch.empty((M, 3), dtype=f32, device=d)
        self.s_flag = torch.empty(M, dtype=torch.uint8, device=d)
        self.feats = torch.empty((M, 16), dtype=f32, device=d)
        self.dfeats = torch.empty((M, 16), dtype=f32, device=d)
        self.sdf = torch.empty(M, dtype=f32, device=d)
        self.act = None
        self._act_key = None
        self.want_decoder_grads = want_decoder_grads
        # fp32 gradient accumulators as views into ONE flat buffer [header(16) | pose_acc F*12 (padded) | grad_emb V*16]: one zero-fill per
        # iteration and, multi-GPU, one all-reduce that also carries the loss sums in the header (dist.allreduce_grads_with_loss)
        self.gradflat = None
        self._gradflat_key = None
        self.grad_emb = None          # fp32 [V,16]
        self.pose_acc = None          # fp32 [F,12]
        self.Rt12 = None
        self.pose_grad = None
        # device-side iteration control block (include/nerfloam_b200.h section 8): sticky error bits, skipped-iteration bookkeeping,
        # Adam's step count -- what lets a whole optimisation call run without a host synchronisation per iteration
        # Two alternating blocks: the decoder's Adam of iteration i may still be running on the side stream while iteration i+1 folds
        # its statistics, so iteration i+1 writes the other block (nl_iter_status copies forward).
        self._ctl2 = torch.zeros((2, _capi.CTL_WORDS), dtype=torch.int32, device=d)
        self._ctl_idx = 0
        self._ctl_init = torch.zeros(_capi.CTL_WORDS, dtype=torch.int32, device=d)
        self._ctl_init[_capi.CTL_MIN_HIT] = 2 ** 31 - 1
        self._ctl2[0].copy_(self._ctl_init)
        self._ctl_host = torch.empty(_capi.CTL_WORDS, dtype=torch.int32).pin_memory() if torch.cuda.is_available() else None
        self._xbuf = None             # packed statistics vector of the multi-GPU exchange
        self._stats_host = torch.empty(STATS_BYTES, dtype=torch.uint8).pin_memory() if torch.cuda.is_available() else None
        self.events = None            # set to {} to record CUDA events around the main kernels (bench.py)
        # the weight-gradient kernels of the decoder run on a second stream, concurrently with the embedding scatter
        self.overlap_wgrad = True
        # warp-cooperative traversal over the packed octree image; False: one thread per ray over (centres, structure)
        self.use_packed_octree = True
        self._side = None
        # software pipelining across iterations (forward_backward(defer_wgrad=True)): the weight-gradient kernels and the decoder's
        # Adam of iteration i stay on the side stream while the main stream already runs the embedding scatter, the other Adam
        # steps and iteration i+1 up to its decoder; what they read of iteration i (sample count, features) is double-buffered
        self._pending = False
        self._alt = None

    def _mark(self, name):
        if self.events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.events.setdefault(name, []).append(ev)

    # ------------------------------------------------------------------ helpers
    @property
    def n_samples_dev(self):
        return C.c_void_p(self.stats.data_ptr() + N_SAMPLES_OFFSET)

    def read_stats(self):
        """Device -> host copy of nl_render_stats (synchronises the stream)."""
        self._stats_host.copy_(self.stats, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return RenderStats.from_buffer_copy(self._stats_host.numpy().tobytes())

    @property
    def ctl(self):
        """The control block of the current iteration (int32[CTL_WORDS] view)."""
        return self._ctl2[self._ctl_idx]

    def begin_call(self):
        """Reset the iteration control block (start of a bundle_adjust_frames / track_frame call)."""
        self.join_side()
        self.ctl.copy_(self._ctl_init)

    def _iter_status(self, alternate):
        prev = self.ctl
        if alternate:
            self._ctl_idx ^= 1
        _capi.check(_capi.lib().nl_iter_status(C.c_void_p(self.stats.data_ptr()), _capi.ptr(prev), _capi.ptr(self.ctl), _capi.stream_ptr()),
                    "nl_iter_status")
        _capi.LAUNCHES += 1

    def read_ctl(self):
        """Device -> host copy of the control block (synchronises the stream): list of CTL_WORDS ints."""
        self._ctl_host.copy_(self.ctl, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._ctl_host.tolist()

    def adopt_gradflat(self, flat, V, n_frames):
        """Use an externally allocated flat gradient buffer of the same layout (dist.PeerReduceAdam's symmetric-memory buffer, so
        that the scatter kernels write where the peers read)."""
        npose = (n_frames * 12 + 15) // 16 * 16
        assert flat.numel() == 16 + npose + V * 16 and flat.dtype == torch.float32 and flat.is_contiguous()
        self.gradflat = flat
        self.pose_acc = flat[16:16 + n_frames * 12].view(n_frames, 12)
        self.grad_emb = flat[16 + npose:].view(V, 16)
        self.pose_grad = torch.zeros((n_frames, 6), dtype=torch.float32, device=self.device)
        self._gradflat_key = (int(V), int(n_frames))

    def _ensure_grads(self, V, n_frames):
        key = (int(V), int(n_frames))
        if self._gradflat_key != key:
            npose = (n_frames * 12 + 15) // 16 * 16
            self.gradflat = torch.zeros(16 + npose + V * 16, dtype=torch.float32, device=self.device)
            self.pose_acc = self.gradflat[16:16 + n_frames * 12].view(n_frames, 12)
            self.grad_emb = self.gradflat[16 + npose:].view(V, 16)
            self.pose_grad = torch.zeros((n_frames, 6), dtype=torch.float32, device=self.device)
            self._gradflat_key = key
            return True
        return False

    def _ensure_act(self, width):
        key = (width, mlp_impl(width))
        if self.act is None or self._act_key != key:
            self.act = alloc_act(width, self.max_samples, self.device)
            self._act_key = key

    # ------------------------------------------------------------------ stages
    def rays_from_poses(self, pose6, dir_local, ray_frame):
        """pose6 f32[F,6] (device), dir_local f32[R,3], ray_frame i32[R] or None -> fills ray_o / ray_d."""
        F, R = pose6.shape[0], dir_local.shape[0]
        if self.Rt12 is None or self.Rt12.shape[0] < F:
            self.Rt12 = torch.empty((F, 12), dtype=torch.float32, device=self.device)
        st = _capi.stream_ptr()
        if F <= 32:      # matrices evaluated inside the ray kernel: one launch
            _capi.check(_capi.lib().nl_rays_from_pose6(R, F, _capi.ptr(dir_local), _capi.ptr(ray_frame), _capi.ptr(pose6), _capi.ptr(self.Rt12),
                                                       _capi.ptr(self.ray_o), _capi.ptr(self.ray_d), st), "nl_rays_from_pose6")
            _capi.LAUNCHES += 1
            return
        _capi.check(_capi.lib().nl_pose_matrices(F, _capi.ptr(pose6), _capi.ptr(self.Rt12), st), "nl_pose_matrices")
        _capi.check(_capi.lib().nl_rays_from_poses(R, _capi.ptr(dir_local), _capi.ptr(ray_frame), _capi.ptr(self.Rt12),
                                                   _capi.ptr(self.ray_o), _capi.ptr(self.ray_d), st), "nl_rays_from_poses")
        _capi.LAUNCHES += 2

    def render_samples(self, m, R, cfg, ray_o=None, ray_d=None, gt_depth=None, cos=None, noise=None, rng_seed=0,
                       reference_compat=True, rng_seed_dev=None):
        """rays -> compact sample list (nl_render_samples).  cfg: dict(voxel_size, step_size, max_distance,
        truncation, max_depth, fs_weight, sdf_weight)."""
        assert R <= self.max_rays
        a = RenderArgs()
        a.n_rays, a.n_nodes, a.sample_capacity, a.reference_compat = R, m.n_nodes, self.max_samples, int(bool(reference_compat))
        a.voxel_size, a.step_size, a.max_distance = cfg["voxel_size"], cfg["step_size"], cfg["max_distance"]
        a.truncation, a.max_depth = cfg.get("truncation", 0.0), cfg.get("max_depth", 0.0)
        a.fs_weight, a.sdf_weight = cfg.get("fs_weight", 0.0), cfg.get("sdf_weight", 0.0)
        a.d_centres, a.d_structure = m.centres.data_ptr(), m.structure.data_ptr()
        a.d_packed_children = m.packed_children().data_ptr() if self.use_packed_octree else None
        a.d_ray_o = (ray_o if ray_o is not None else self.ray_o).data_ptr()
        a.d_ray_d = (ray_d if ray_d is not None else self.ray_d).data_ptr()
        a.d_gt_depth = gt_depth.data_ptr() if gt_depth is not None else None
        a.d_cos = cos.data_ptr() if cos is not None else None
        if noise is not None:
            assert noise.is_cuda and noise.dtype == torch.float32 and noise.is_contiguous() and noise.dim() == 2
            a.d_noise, a.noise_stride = noise.data_ptr(), noise.shape[1]
        a.rng_seed = int(rng_seed) & 0xffffffff
        a.d_rng_seed = rng_seed_dev.data_ptr() if rng_seed_dev is not None else None   # int32 tensor on the device (CUDA-graph replays)
        a.d_workspace, a.workspace_bytes = self.workspace.data_ptr(), self.ws_bytes
        a.d_stats, a.d_hit_rank = self.stats.data_ptr(), self.hit_rank.data_ptr()
        a.d_s_ray, a.d_s_vox, a.d_s_depth = self.s_ray.data_ptr(), self.s_vox.data_ptr(), self.s_depth.data_ptr()
        a.d_s_xyz, a.d_s_flag = self.s_xyz.data_ptr(), self.s_flag.data_ptr()
        a.d_ray_nsamp, a.d_ray_offset = self.ray_nsamp.data_ptr(), self.ray_offset.data_ptr()
        _capi.check(_capi.lib().nl_render_samples(C.byref(a), _capi.stream_ptr()), "nl_render_samples")
        _capi.LAUNCHES += 6 if gt_depth is not None else 5

    def gather_forward(self, m, M_cap=None, xyz=None, vox=None, M_dev=True, feats=None):
        M_cap = self.max_samples if M_cap is None else M_cap
        _capi.check(_capi.lib().nl_gather_trilinear_fwd(
            M_cap, self.n_samples_dev if M_dev else None, _capi.ptr(xyz if xyz is not None else self.s_xyz),
            _capi.ptr(vox if vox is not None else self.s_vox), _capi.ptr(m.centres), _capi.ptr(m.vox2row), _capi.ptr(m.emb),
            float(self._vs), _capi.ptr(feats if feats is not None else self.feats), _capi.stream_ptr()), "nl_gather_trilinear_fwd")
        _capi.LAUNCHES += 1

    # ------------------------------------------------------------------ full passes
    def side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def deferred_stream(self):
        """The side stream if the last forward_backward(defer_wgrad=True) left decoder work on it (pass it to
        FusedAdam.step(side_stream=...) so the decoder's update follows its gradients there), else None."""
        return self._side if self._pending else None

    def join_side(self):
        """Main stream waits for deferred decoder work (weight gradients + the decoder's Adam) of the previous iteration."""
        if self._pending:
            torch.cuda.current_stream(self.device).wait_stream(self._side)
            self._pending = False

    def _flip_buffers(self):
        if self._alt is None:
            self._alt = (torch.zeros_like(self.stats), torch.empty_like(self.feats))
        (self.stats, self.feats), self._alt = self._alt, (self.stats, self.feats)

    def forward(self, m, dec, R, cfg, ray_o=None, ray_d=None, noise=None, rng_seed=0, reference_compat=True):
        """Forward only (render_rays / evaluation): fills s_*, feats, sdf.  Returns nothing; read_stats() for sizes."""
        self.join_side()
        self._vs = cfg["voxel_size"]
        self.render_samples(m, R, cfg, ray_o, ray_d, None, None, noise, rng_seed, reference_compat)
        dec.refresh_transposes()
        self.gather_forward(m)
        mlp_forward(dec, self.max_samples, self.n_samples_dev, self.feats, self.sdf)

    def forward_backward(self, m, dec, R, cfg, gt_depth, cos, dir_local=None, ray_frame=None, n_frames=1, ray_o=None,
                         ray_d=None, noise=None, rng_seed=0, reference_compat=True, update_decoder=True, update_emb=True,
                         update_pose=True, pose6=None, group=None, refresh_weights=True, rng_seed_dev=None, defer_wgrad=False, peer=None,
                         peer_stats=None, pose_step=None):
        """One optimisation iteration without the optimiser step.  Gradients land in
        self.grad_emb (fp32 [V,16]), dec.grads (fp32), self.pose_grad (fp32 [F,6]); the loss in stats.
        defer_wgrad=True: return without waiting for the decoder's weight gradients -- they (and whatever the caller enqueues on
        side_stream(), i.e. the decoder's optimiser step) are joined right before the next iteration's decoder, or by join_side().
        pose_step: dict(mask, m, v, lr, seeds=[(int32 tensor, increment), ...]) -- the pose gradient, the poses' Adam step (rows in
        `mask`, moments m / v f32[F,6]), the loss read-out and the advance of the listed device-side seeds as ONE launch
        (nl_pose_step) instead of nl_pose_grad + nl_loss_finalize + one Adam launch per pose + one add per seed."""
        lib = _capi.lib()
        st = _capi.stream_ptr()
        self._vs = cfg["voxel_size"]
        if self._pending:
            self._flip_buffers()     # the deferred kernels still read the previous iteration's sample count and features
        self._mark("t0")
        self.render_samples(m, R, cfg, ray_o, ray_d, gt_depth, cos, noise, rng_seed, reference_compat, rng_seed_dev)
        if group is not None:   # the loss normalisation is global (criterion.py:84-100): ONE tiny exchange before backward
            from . import dist as nldist
            if peer_stats is not None:      # through symmetric memory on this stream: pack, barrier, sum of the peers' vectors
                peer_stats.exchange(self.stats, cfg["fs_weight"], cfg["sdf_weight"])
            else:
                self._xbuf = nldist.allreduce_sample_stats(self.stats, group, self._xbuf, cfg["fs_weight"], cfg["sdf_weight"])
        self._iter_status(alternate=defer_wgrad)      # captured CUDA graphs (tracking) keep one block: fixed pointers
        self._mark("t_samples")
        if peer is not None:
            peer.wait_params()       # the previous iteration's table slices of every rank have landed (barrier deferred to here)
        self.gather_forward(m)
        self.join_side()             # decoder weights (and gradient buffers) of the previous iteration are final from here on
        if refresh_weights:
            dec.refresh_transposes()
        self._mark("t_gather_fwd")
        if update_decoder:
            self._ensure_act(dec.width)
            dec.gradflat.zero_()
        side = None
        if update_decoder and self.overlap_wgrad and mlp_impl(dec.width) == "tc":
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)
            side = self._side
        mlp_train(dec, self.max_samples, self.n_samples_dev, self.feats, self.sdf, self.dfeats, update_decoder, self.act,
                  s_flag=self.s_flag, s_depth=self.s_depth, s_ray=self.s_ray, cos=cos, gt_depth=gt_depth,
                  stats_ptr=C.c_void_p(self.stats.data_ptr()), truncation=cfg["truncation"], wgrad_stream=side)
        self._mark("t_mlp")
        want_pose = update_pose and dir_local is not None
        if update_emb or want_pose:
            if not self._ensure_grads(m.emb.shape[0] if update_emb else 0, n_frames):
                self.gradflat.zero_()
        if update_emb or want_pose:
            _capi.check(lib.nl_gather_trilinear_bwd(
                self.max_samples, self.n_samples_dev, _capi.ptr(self.s_xyz), _capi.ptr(self.s_vox), _capi.ptr(m.centres),
                _capi.ptr(m.vox2row), _capi.ptr(m.emb), float(cfg["voxel_size"]), _capi.ptr(self.dfeats), 1,
                _capi.ptr(self.grad_emb) if update_emb else None, None, _capi.ptr(self.s_ray), _capi.ptr(self.s_depth),
                _capi.ptr(dir_local) if want_pose else None, _capi.ptr(ray_frame) if want_pose else None, int(n_frames),
                _capi.ptr(self.pose_acc) if want_pose else None, st), "nl_gather_trilinear_bwd")
            _capi.LAUNCHES += 1
        defer = defer_wgrad and side is not None
        if side is not None and not defer:
            torch.cuda.current_stream(self.device).wait_stream(side)   # decoder gradients complete before they are reduced / applied
        self._mark("t_gather_bwd")
        if group is not None:
            from . import dist as nldist
            if self.gradflat is None:
                self._ensure_grads(0, n_frames)
            if peer is not None:     # fused reduce-scatter -> Adam -> all-gather over NVLink peer memory (the table's Adam step is inside)
                peer.step(self.stats, self.ctl, self.pose_acc if want_pose else None, defer_barrier=True)
            else:
                nldist.allreduce_grads_with_loss(self.stats, self.gradflat, group)     # loss sums + pose accumulators + embedding gradients
            if update_decoder:       # the decoder's gradients are reduced where they are produced
                with (torch.cuda.stream(side) if defer else contextlib.nullcontext()):
                    nldist.allreduce_flat(dec.gradflat, group)
        if defer:
            self._pending = True
        if pose_step is not None and want_pose and n_frames <= 31:
            seeds = list(pose_step.get("seeds", ())) + [(None, 0), (None, 0)]
            _capi.check(lib.nl_pose_step(n_frames, _capi.ptr(pose6), _capi.ptr(self.pose_acc), _capi.ptr(self.pose_grad), int(pose_step["mask"]),
                                         _capi.ptr(pose_step["m"]), _capi.ptr(pose_step["v"]), float(pose_step["lr"]), 0.9, 0.999, 1e-8,
                                         _capi.ptr(self.ctl), C.c_void_p(self.stats.data_ptr()), float(cfg["fs_weight"]), float(cfg["sdf_weight"]),
                                         _capi.ptr(seeds[0][0]), int(seeds[0][1]), _capi.ptr(seeds[1][0]), int(seeds[1][1]), st), "nl_pose_step")
            _capi.LAUNCHES += 1
            return
        if want_pose:
            _capi.check(lib.nl_pose_grad(n_frames, _capi.ptr(pose6), _capi.ptr(self.pose_acc), _capi.ptr(self.pose_grad), st),
                        "nl_pose_grad")
            _capi.LAUNCHES += 1
        _capi.check(lib.nl_loss_finalize(C.c_void_p(self.stats.data_ptr()), float(cfg["fs_weight"]), float(cfg["sdf_weight"]), st),
                    "nl_loss_finalize")
        _capi.LAUNCHES += 1


class FusedAdam:
    """torch.optim.Adam semantics (fresh state per construction, like render_helpers.py:353 / :448) with one
    fused kernel per tensor.  groups: list of dict(param=tensor, grad=tensor(fp32), lr=float).
    ctl: the engine's device-side iteration control block (SDFEngine.ctl, or a callable returning the current one).  With it the step count lives on the device and an
    iteration the reference would have skipped (no hits: `continue` before optim.step(), render_helpers.py:405-409) leaves
    parameters, moments and the step count untouched -- without a host synchronisation."""

    def __init__(self, groups, betas=(0.9, 0.999), eps=1e-8, ctl=None):
        self.groups = groups
        self.betas, self.eps = betas, eps
        self.step_count = 0
        self.ctl = ctl
        for g in groups:
            p = g["param"]
            g["m"] = torch.zeros_like(p)
            g["v"] = torch.zeros_like(p)
        # the moments are zero-filled on the constructing stream; a side stream that updates some of the groups has to be ordered
        # behind that (its only other dependency is the decoder kernel of the iteration, enqueued BEFORE this constructor ran)
        self._init_event = None
        if any(g.get("side") for g in groups) and groups[0]["param"].is_cuda:
            self._init_event = torch.cuda.Event()
            self._init_event.record(torch.cuda.current_stream(groups[0]["param"].device))

    def step(self, side_stream=None):
        """side_stream: the groups marked side=True (the decoder, whose gradients are produced there) are updated on that stream."""
        self.step_count += 1
        lib = _capi.lib()
        if side_stream is not None and self._init_event is not None:
            side_stream.wait_event(self._init_event)
            self._init_event = None
        passes = [(None, self.groups)] if side_stream is None else \
            [(None, [g for g in self.groups if not g.get("side")]), (side_stream, [g for g in self.groups if g.get("side")])]
        for stream, gs in passes:
            with (torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()):
                st = _capi.stream_ptr()
                for g in gs:
                    p = g["param"]
                    bf = p.dtype == torch.bfloat16
                    if self.ctl is not None:
                        fn = lib.nl_adam_bf16_ctl if bf else lib.nl_adam_f32_ctl
                        last = _capi.ptr(self.ctl() if callable(self.ctl) else self.ctl)
                    else:
                        fn = lib.nl_adam_bf16 if bf else lib.nl_adam_f32
                        last = self.step_count
                    _capi.check(fn(p.numel(), _capi.ptr(p), _capi.ptr(g["grad"]), _capi.ptr(g["m"]), _capi.ptr(g["v"]), float(g["lr"]),
                                   self.betas[0], self.betas[1], self.eps, last, st), "nl_adam")
                    _capi.LAUNCHES += 1
