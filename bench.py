#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native NeRF-LOAM hot path (BASELINE.json metric):
neural-SDF samples/s per mapping iteration on a synthetic 100k-ray KITTI-shape scan.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one full mapping iteration of bundle_adjust_frames' loop body on every ray of one scan per GPU:
pose -> rays -> octree traversal -> inverse-CDF sampling -> embedding gather + trilinear -> 16-256-256-1 MLP
-> SDF/free-space loss -> backward (decoder, embeddings, pose) -> Adam on all three.  Prints ONE JSON line.

--dump-outputs DIR writes what the last of the K timed steps hands back to its caller -- the embedding table, decoder and pose
after Adam, and the loss -- as DIR/<name>.npy, arrays whose shapes depend only on the arguments.  The timed steps start from the
seeded problem as built, so two builds run with the same arguments can be compared output for output; what differs between two
runs of one build is the order of float atomics within those K steps, which a mapping loop amplifies (the pose gradient is a sum
of ~10^5 cancelling terms, and the pose moves the rays: the number of samples, hence the per-sample SDF, is not dumped because
its length differs by a few samples in 775k from run to run).  Measured on a B200: with --steps 1 two runs give the same loss bit
for bit and the same parameters up to one bf16 rounding step of the table; with --steps 20 the parameters agree to ~2e-3
relative norm.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(step_size=0.5 * 0.3, voxel_size=0.3, max_distance=40.0, truncation=0.3, max_depth=40.0, fs_weight=1.0, sdf_weight=10000.0)
LR = (0.01, 0.005, 0.001)                     # kitti.yaml learning_rate_emb / _decorder / _pose
BYTES_PER_SAMPLE_MAP = 1116                   # BASELINE.md: algorithmic HBM bytes / valid sample, MAP mode
FLOPS_PER_SAMPLE_MAP_DEC = 419328             # BASELINE.md: MLP fwd + bwd-data + bwd-weight
# tf32 tensor-core FLOPs actually issued per sample for that fp32-parity result: 3 terms (hi*hi, hi*lo, lo*hi) for layer 1/2
# forward, backward layer 1 and gW0|gb0 (N = 32); 2 terms for backward layer 2 and gW1 (one operand is the exact 0/1 ReLU mask)
ISSUED_TF32_FLOPS_PER_SAMPLE = 2 * (3 * 16 * 256 + 3 * 256 * 256 + 2 * 256 * 256 + 3 * 256 * 16 + 2 * 256 * 256 + 3 * 256 * 32)
WORKLOAD = "synthetic 100k-ray KITTI-shape scan (64x1563 beams, 82.7k returns), single-scan 0.3 m map, " \
           "mapping iteration on ALL rays, decoder+embeddings+pose updated, Adam included"
# untimed steps between the warm-up and the clock, so that clocks, allocator, NCCL channels and the two-stream pipeline reach
# steady state (64 steps took ~100 ms on a B200).  A fixed count, not a duration: the state the timed steps start from must not
# depend on how fast the machine is
SETTLE_STEPS = 64


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(gpu)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_problem(nl, n_maps_scans, device):
    """Replicated map from `n_maps_scans` scans (deterministic, identical on every rank)."""
    syn = nl.synthetic
    scans = [syn.make_scan(seed=777 + i) for i in range(n_maps_scans)]
    mu = nl.mapping.MapUpdater(CFG["voxel_size"], init_std=0.01, seed=777, device=device)
    for pts, cos, pose in scans:
        mu.svo.insert(torch.from_numpy(syn.voxelize(pts, pose, CFG["voxel_size"])))
    ms = mu.update_grid_features()
    torch.manual_seed(777)
    dec = nl.lidar.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).to(device)
    return scans, mu, ms, dec


def host_rays(pts, cos):
    P = torch.from_numpy(pts)
    dirs = (P / (P.norm(dim=-1, keepdim=True) + 1e-8)).float().contiguous()
    gt = (torch.norm(P, 2, -1) * torch.from_numpy(cos)).float().contiguous()
    return dirs.pin_memory(), gt.pin_memory(), torch.from_numpy(cos).float().contiguous().pin_memory()


def _traffic_record(kernel_key):
    """dram bytes per launch of the dominant kernel from the committed ncu capture of THIS build (profiles/r02_traffic.json, written by
    scripts/summarise_profiles.py from an `ncu --set full` report); None when no capture is recorded."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    rec = d.get(kernel_key)
    if not rec:
        return None, None
    return rec.get("dram_bytes"), {"ncu_report": rec.get("report"), "read": rec.get("read"), "write": rec.get("write"), "samples": rec.get("samples")}


def run_ours(args):
    import nerfloam_b200 as nl
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    # ONE clock poller for the whole job, started before the warm-up (eight NVML attaches right before the timed region were a
    # transient inside it in round 1)
    clocks = ClockSampler(local) if rank == 0 else None
    scans, mu, ms, dec = build_problem(nl, world, dev)
    pts, cos, pose = scans[rank]
    h_dirs, h_gt, h_cos = host_rays(pts, cos)
    R = h_dirs.shape[0]
    d_dirs, d_gt, d_cos = h_dirs.to(dev), h_gt.to(dev), h_cos.to(dev)
    pose6 = nl.se3pose.OptimizablePose.from_matrix(torch.from_numpy(pose)).data.detach().reshape(1, 6).to(dev).contiguous()
    eng = nl.engine.SDFEngine(R, R * 20, dev)
    bufs = nl.engine.DecoderBuffers(dec, dev)
    emb = ms.emb
    state = {"opt": None}
    # multi-GPU: the embedding-gradient reduction fused with the table's Adam step over NVLink peer memory (csrc/peer.cu) and the
    # statistics exchange through symmetric memory, instead of NCCL all-reduces (NL_PEER=0: plain NCCL, the baseline)
    peer = pstats = None
    peer_info = None
    if world > 1 and os.environ.get("NL_PEER", "1") != "0":
        try:
            peer = nl.dist.PeerReduceAdam(group, dev, emb.shape[0], 1, lr=LR[0])
            peer.param.copy_(emb)
            ms = nl.engine.MapState(ms.centres, ms.structure, ms.vox2row, peer.param, dev)
            emb = ms.emb
            eng.adopt_gradflat(peer.grad, emb.shape[0], 1)
            pstats = nl.dist.PeerStats(group, dev)
            peer_info = {"fused_reduce_adam": True, "nvls_multicast": peer.multicast}
        except Exception as exc:      # no symmetric memory on this system: NCCL path
            peer = pstats = None
            peer_info = {"fused_reduce_adam": False, "why": repr(exc)}

    pipeline = os.environ.get("NL_PIPELINE", "1") != "0"

    def step(dirs, gt, cosv, update_decoder=True):
        eng.rays_from_poses(pose6, dirs, None)
        eng.forward_backward(ms, bufs, R, CFG, gt, cosv, dir_local=dirs, ray_frame=None, n_frames=1, rng_seed=12345,
                             update_decoder=update_decoder, update_emb=True, update_pose=True, pose6=pose6, group=group,
                             defer_wgrad=pipeline and update_decoder and eng.overlap_wgrad, peer=peer, peer_stats=pstats)
        emb_group = [] if peer is not None else [dict(param=emb, grad=eng.grad_emb, lr=LR[0])]      # peer: the table's Adam is inside the fused kernel
        if not update_decoder:          # steady-state variant (decoder frozen after freeze_frame frames, mapping.py:196)
            if "opt_frozen" not in state:
                state["opt_frozen"] = nl.engine.FusedAdam(emb_group + [dict(param=pose6[0], grad=eng.pose_grad[0], lr=LR[2])], ctl=lambda: eng.ctl)
            state["opt_frozen"].step()
            return
        if state["opt"] is None:
            state["opt"] = new_opt(emb_group)
        # pipelined: the decoder's Adam follows its weight-gradient kernels on the side stream; the main stream goes on with the
        # embedding / pose update and the next iteration's rays, traversal, sampling and gather, and joins before its decoder
        state["opt"].step(side_stream=eng.deferred_stream())

    def new_opt(emb_group):
        groups = list(emb_group)
        groups += [dict(param=p.data, grad=g, lr=LR[1], side=True) for p, g in zip(bufs.params, bufs.grads)]
        groups += [dict(param=pose6[0], grad=eng.pose_grad[0], lr=LR[2])]
        return nl.engine.FusedAdam(groups, ctl=lambda: eng.ctl)

    def sync_all():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, finish=None):
        """n calls of fn between two events (barrier + synchronize on both sides): total ms."""
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        if finish:
            finish()
        b.record()
        sync_all()
        return a.elapsed_time(b)

    # ---------------- device-resident timing (value) ----------------
    # the timed steps start from the problem as built, not from what the warm-up and settle steps left: those accumulate gradients
    # with float atomics, so their result differs in the last bits from run to run, and Adam amplifies that step after step
    start = [t.detach().clone() for t in [emb, pose6] + bufs.params]
    eng.begin_call()
    W = max(args.warmup, 3)
    for _ in range(W):
        step(d_dirs, d_gt, d_cos)
    for i in range(SETTLE_STEPS):
        step(d_dirs, d_gt, d_cos)
        if i % 8 == 7:
            torch.cuda.synchronize()
    eng.join_side()
    sync_all()                                         # multi-GPU: no peer still reads this rank's table
    with torch.no_grad():
        for t, t0 in zip([emb, pose6] + bufs.params, start):
            t.copy_(t0)
        if peer is not None:
            peer.m.zero_(); peer.v.zero_()
    eng.begin_call()                                   # Adam's step count
    state["opt"] = new_opt([] if peer is not None else [dict(param=emb, grad=eng.grad_emb, lr=LR[0])])
    l0 = nl._capi.LAUNCHES
    ms_total = timed(lambda: step(d_dirs, d_gt, d_cos), args.steps, eng.join_side)   # deferred decoder work of the last iteration is inside
    launches = nl._capi.LAUNCHES - l0
    st = eng.read_stats()
    n_local = st.n_samples
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st, dec, emb, pose6)
    # ---------------- the same loop over >= 250 ms with one event per step: median / max (what a 32 ms window cannot show) ----------------
    n_long = max(args.steps, int(0.25 / max(ms_total / args.steps * 1e-3, 1e-6)) + 1)
    if world > 1:
        import torch.distributed as dist
        t_n = torch.tensor([n_long], device=dev); dist.all_reduce(t_n, op=dist.ReduceOp.MAX); n_long = int(t_n.item())
    sync_all()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_long + 1)]
    evs[0].record()
    for i in range(n_long):
        step(d_dirs, d_gt, d_cos)
        evs[i + 1].record()
    eng.join_side()
    sync_all()
    per_step = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(n_long)])
    long_stats = {"steps": n_long, "ms_total": float(evs[0].elapsed_time(evs[-1])), "ms_median": float(np.median(per_step)),
                  "ms_p90": float(np.percentile(per_step, 90)), "ms_max": float(per_step.max()), "ms_mean": float(per_step.mean())}
    # per-stage times for the roofline: a separate pass with CUDA events around the stages and the weight-gradient kernels
    # serialised on the main stream (in the timed loop above they overlap with the embedding scatter on a second stream)
    ov = eng.overlap_wgrad
    eng.overlap_wgrad = False
    step(d_dirs, d_gt, d_cos)
    sync_all()
    eng.events = {}
    for _ in range(args.steps):
        step(d_dirs, d_gt, d_cos)
    sync_all()
    ev = eng.events
    eng.events = None
    eng.overlap_wgrad = ov
    t_mlp = float(np.mean([a.elapsed_time(b) for a, b in zip(ev["t_gather_fwd"], ev["t_mlp"])]))
    t_gf = float(np.mean([a.elapsed_time(b) for a, b in zip(ev["t_samples"], ev["t_gather_fwd"])]))
    t_gb = float(np.mean([a.elapsed_time(b) for a, b in zip(ev["t_mlp"], ev["t_gather_bwd"])]))
    t_smp = float(np.mean([a.elapsed_time(b) for a, b in zip(ev["t0"], ev["t_samples"])]))

    # ---------------- secondary: steady-state mapping iteration with the decoder frozen ----------------
    for _ in range(3):
        step(d_dirs, d_gt, d_cos, update_decoder=False)
    sync_all()
    eng.events = {}
    ms_frozen = timed(lambda: step(d_dirs, d_gt, d_cos, update_decoder=False), args.steps, eng.join_side)
    evf = eng.events
    eng.events = None
    t_mlp_frozen = float(np.mean([a.elapsed_time(b) for a, b in zip(evf["t_gather_fwd"], evf["t_mlp"])]))

    # ---------------- secondary metric of BASELINE.json: tracking ms/scan through the drop-in track_frame ----------------
    track = None
    if world == 1 and not os.environ.get("NL_BENCH_SKIP_TRACKING"):
        try:
            from types import SimpleNamespace
            crit = nl.criterion.Criterion(SimpleNamespace(criteria={"eiko_weight": 0.1, "sdf_weight": CFG["sdf_weight"], "fs_weight": CFG["fs_weight"],
                                                                   "sdf_truncation": CFG["truncation"]}, data_specs={"max_depth": CFG["max_depth"]}))
            fr = nl.frame.LidarFrame(5, torch.from_numpy(pts), torch.from_numpy(cos), nl.se3pose.OptimizablePose(pose6[0].detach().cpu().clone()),
                                     new_keyframe=True)
            torch.manual_seed(1)
            def one_scan(mode):
                return nl.render_helpers.track_frame(fr.pose, fr, ms, dec, crit, CFG["voxel_size"], N_rays=2048, step_size=0.2 * CFG["voxel_size"],
                                                     num_iterations=25, truncation=CFG["truncation"], learning_rate=0.06, max_voxel_hit=20,
                                                     max_distance=CFG["max_distance"], ray_selection="host" if mode == "host" else "device",
                                                     cuda_graph=(mode == "graph"))
            res = {}
            for mode, nscan in (("host", 3), ("device", 10), ("graph", 10)):
                one_scan(mode)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(nscan):
                    one_scan(mode)
                torch.cuda.synchronize()
                res[mode] = (time.perf_counter() - t0) / nscan * 1e3
            track = {"ms_per_scan": min(res["device"], res["graph"]), "ms_per_scan_cuda_graph": res["graph"], "ms_per_scan_eager": res["device"],
                     "ms_per_scan_host_selection": res["host"], "iterations": 25, "rays_per_iteration": 2048,
                     "note": "track_frame() drop-in, wall clock per 25-iteration scan.  eager: ray_selection='device' (uniform without "
                             "replacement drawn on the GPU), one stats read-back per iteration; cuda_graph: the iteration captured once per "
                             "scan and replayed 24x, one read-back per scan; host_selection: the reference's per-iteration CPU Gumbel top-k "
                             "over all points of the scan (frame.sample_rays), which dominates it"}
        except Exception as exc:   # never let the secondary metric break the headline line
            track = {"error": repr(exc)}

    # ---------------- end-to-end through the public step with host buffers (e2e) ----------------
    loss_host = torch.empty(nl.engine.STATS_BYTES, dtype=torch.uint8).pin_memory()
    s_dirs, s_gt, s_cos = torch.empty_like(d_dirs), torch.empty_like(d_gt), torch.empty_like(d_cos)

    def step_e2e():
        s_dirs.copy_(h_dirs, non_blocking=True); s_gt.copy_(h_gt, non_blocking=True); s_cos.copy_(h_cos, non_blocking=True)
        step(s_dirs, s_gt, s_cos)
        loss_host.copy_(eng.stats, non_blocking=True)
    for _ in range(3):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps, eng.join_side)
    loss_val = nl._capi.RenderStats.from_buffer_copy(loss_host.numpy().tobytes()).loss
    ctl = eng.read_ctl()

    # ---------------- north-star split (BASELINE.json config 5): ONE scan ray-sharded over the ranks (strong scaling) ----------------
    strong = None
    if world > 1:
        if peer is not None:
            peer.wait_params()
        strong = strong_scaling_block(nl, dev, rank, world, group, scans[0], ms, dec, args.steps, sync_all, timed, use_peer=peer is not None)

    clk = clocks.stop() if clocks is not None else None

    # ---------------- aggregate over ranks (max time, sum samples) ----------------
    t = torch.tensor([ms_total, ms_e2e, float(n_local), long_stats["ms_total"], long_stats["ms_median"], long_stats["ms_max"]], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        ms_total, ms_e2e, n_total = float(tm[0]), float(tm[1]), float(ts[2])
        long_stats.update(ms_total=float(tm[3]), ms_median=float(tm[4]), ms_max=float(tm[5]), note="max over ranks")
    else:
        n_total = float(n_local)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    pk = peaks()
    value = n_total * args.steps / (ms_total * 1e-3)
    e2e = n_total * args.steps / (ms_e2e * 1e-3)
    flops = n_local * FLOPS_PER_SAMPLE_MAP_DEC
    ach_tf = flops / (t_mlp * 1e-3) / 1e12
    gather_gbs = n_local * BYTES_PER_SAMPLE_MAP / ((t_gf + t_gb) * 1e-3) / 1e9
    tc = nl.engine.mlp_impl(256) == "tc"
    traffic, traffic_src = _traffic_record("k_mlp_tc_train" if tc else "k_mlp")
    long_stats["value_from_median"] = n_total / (long_stats["ms_median"] * 1e-3)
    out = {
        "metric": "neural-SDF samples/sec per mapping iter", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_gpu": R, "samples_per_gpu_step": n_local, "octree_nodes": ms.n_nodes,
                   "embedding_rows": int(ms.emb.shape[0]), "decoder": "16-256-256-1, fp32 parity (%s)" % nl.engine.mlp_impl(256),
                   "parallelism": f"ray-sharded dp{world}, map replicated" + ("" if world == 1 else
                                  f": the batch is a window of {world} scans (all rays), split contiguously = one scan per rank; per step: statistics exchange, "
                                  "embedding-gradient reduction (fused with Adam over NVLink peer memory when multi_gpu_exchange.fused_reduce_adam), "
                                  "decoder-gradient all-reduce (NCCL, side stream)"),
                   "l2": "per-step working set (samples x ~2.2 KB activations+features) ~1.9 GB >> 126 MB L2; no flush needed",
                   "sampler_noise": "in-kernel counter RNG", "loss": loss_val,
                   "untimed_before_clock": f"{W} warm-up steps + {SETTLE_STEPS} settle steps, then parameters and Adam state reset to the seeded start",
                   "kernel_error_bits_over_all_steps": ctl[nl._capi.CTL_ERROR], "skipped_steps": ctl[nl._capi.CTL_SKIPPED],
                   "multi_gpu_exchange": peer_info},
        "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": int(R * 20 * world), "d2h_bytes_per_step": int(160 * world),
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "steady_state": long_stats,
        "roofline": {"bound": "tensor",
                     "kernel": ("tc::k_mlp_tc_train<wgrad> + tc::k_dw1_tc + tc::k_dw0_tc (+ k_mask_colsum) (tcgen05.mma kind::tf32, 3-term hi/lo split; 2 terms where "
                                "one operand is the exact 0/1 ReLU mask)"
                                if tc else "k_mlp<256,train,wgrad> + k_dw1 (fp32 CUDA-core FMA)"),
                     "achieved": ach_tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach_tf / pk["bf16_sustained"],
                     "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": pk["src"] + " dense bf16 cuBLAS (sustained).  The fp32-parity path runs on kind::tf32 (half the bf16 rate); a "
                                    "pure 3xTF32 evaluation (3 passes everywhere) could reach at most 1/6 of this peak = %.0f TFLOP/s of algorithmic "
                                    "fp32 FLOPs; two of the five GEMMs here need only 2 passes (exact 0/1 mask operand), so that figure is a "
                                    "reference point, not a ceiling -- tf32_pipe below is the fraction of the tf32 peak actually issued" % (pk["bf16_sustained"] / 6),
                     "vs_pure_3xtf32": ach_tf / (pk["bf16_sustained"] / 6),
                     "tf32_pipe": {"issued_flops_per_sample": ISSUED_TF32_FLOPS_PER_SAMPLE,
                                   "achieved": n_local * ISSUED_TF32_FLOPS_PER_SAMPLE / (t_mlp * 1e-3) / 1e12,
                                   "peak": pk["bf16_sustained"] / 2, "unit": "TFLOP/s",
                                   "frac": n_local * ISSUED_TF32_FLOPS_PER_SAMPLE / (t_mlp * 1e-3) / 1e12 / (pk["bf16_sustained"] / 2),
                                   "note": "the 'sustained' cuBLAS peak was measured power-capped at ~1380 MHz while these kernels run at ~1965 MHz; "
                                           "the clock-independent figure is ncu's sm__pipe_tensor_cycles_active (profiles/)"},
                     "ms_per_launch": t_mlp, "algorithmic_flops_per_sample": FLOPS_PER_SAMPLE_MAP_DEC},
        "roofline_gather": {"bound": "hbm", "kernel": "k_gather_fwd + k_gather_bwd", "achieved": gather_gbs, "peak": pk["hbm"], "unit": "GB/s",
                            "frac": gather_gbs / pk["hbm"], "ms_fwd": t_gf, "ms_bwd": t_gb, "algorithmic_bytes_per_sample": BYTES_PER_SAMPLE_MAP,
                            "note": "ALGORITHMIC bytes (no credit for cache reuse) over the HBM copy peak: an efficiency proxy.  The single-scan "
                                    "table (0.8 MB) is L2-resident, so the DRAM traffic of these kernels is far below this figure (ncu: "
                                    "gpu__dram_throughput ~6 %) -- not an HBM measurement"},
        "roofline_chain": {"bound": "hbm", "what": "whole step against the north star's HBM-gather roofline", "achieved": value / world * BYTES_PER_SAMPLE_MAP / 1e9,
                           "peak": pk["hbm"], "unit": "GB/s", "frac": value / world * BYTES_PER_SAMPLE_MAP / 1e9 / pk["hbm"]},
        "stage_ms": {"traverse_sample": t_smp, "gather_fwd": t_gf, "mlp_fwd_bwd": t_mlp, "gather_bwd": t_gb,
                     "note": "separate pass, stages serialised on one stream; in the timed loop the weight-gradient kernels run on a "
                             "second stream concurrently with the embedding scatter (overlap_wgrad=%s)" % eng.overlap_wgrad},
        "frozen_decoder": {"value": n_local * args.steps / (ms_frozen * 1e-3), "unit": "samples/s (this rank)", "ms_per_step": ms_frozen / args.steps,
                           "mlp_fwd_bwd_ms": t_mlp_frozen,
                           "note": "same iteration with update_decoder=False (steady state after freeze_frame frames, mapping.py:196)"},
        "clocks": clk,
        "tracking": track,
    }
    if strong is not None:
        out["strong_scaling"] = strong
    if world == 1 and not os.environ.get("NL_BENCH_SKIP_REFGPU"):
        # Baseline B + the drop-in at the reference's real iteration size, after every timed region of the product
        try:
            syn = nl.synthetic
            window = [syn.make_scan(seed=777 + i, sensor_xyz=(1.0 * i, 0.0, 0.0)) for i in range(5)]     # config 2: 1 m spacing along +x
            mu_w = nl.mapping.MapUpdater(CFG["voxel_size"], init_std=0.01, seed=777, device=dev)
            for p_, c_, T_ in window:
                mu_w.svo.insert(torch.from_numpy(syn.voxelize(p_, T_, CFG["voxel_size"])))
            ms_w = mu_w.update_grid_features()
            torch.manual_seed(777)
            dec_w = nl.lidar.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).to(dev)
            out["real_size"] = ours_real_size(nl, dev, window, ms_w, dec_w)
            del mu_w, ms_w, dec_w
            torch.cuda.empty_cache()
            rg = reference_gpu(nl, dev, args.steps, scans[0], window)
            out["reference_gpu"] = rg
            if "full_scan_iteration" in rg:
                rg["speedup"] = {"samples_per_s_e2e_vs_reference": e2e / rg["full_scan_iteration"]["samples_per_s"],
                                 "traverse_sample_front_end_vs_reference_kernels": (rg["kernels"]["svo_intersect_ms"] + rg["kernels"]["inverse_cdf_sampling_ms"]) / t_smp,
                                 "bundle_adjust_frames_5x2048x25": rg["bundle_adjust_frames_5x2048x25"]["ms_per_call"] / out["real_size"]["ms_per_call_host_selection"],
                                 "bundle_adjust_frames_5x2048x25_device_selection": rg["bundle_adjust_frames_5x2048x25"]["ms_per_call"] / out["real_size"]["ms_per_call_device_selection"],
                                 "bundle_adjust_frames_5x2048x25_cuda_graph": rg["bundle_adjust_frames_5x2048x25"]["ms_per_call"] / out["real_size"]["ms_per_call_cuda_graph"],
                                 "track_frame_2048x25": (rg["track_frame_2048x25"]["ms_per_scan"] / track["ms_per_scan_host_selection"]) if track and "ms_per_scan" in track else None,
                                 "track_frame_2048x25_cuda_graph": (rg["track_frame_2048x25"]["ms_per_scan"] / track["ms_per_scan_cuda_graph"]) if track and "ms_per_scan" in track else None}
        except Exception as exc:
            out["reference_gpu"] = {"error": repr(exc)}
    if world == 1 and not os.environ.get("NL_BENCH_SKIP_CONFIGS"):
        try:
            out["configs"] = configs_real_size(nl, dev)
        except Exception as exc:
            out["configs"] = {"error": repr(exc)}
    if world == 1 and not os.environ.get("NL_BENCH_SKIP_CPU"):
        out["cpu_baseline"] = best_cpu_baseline(n_rays=4096, iters=3)
    print(json.dumps(out))


def dump_outputs(out_dir, st, dec, emb, pose6):
    """What the last timed step hands back, as out_dir/<name>.npy: the embedding table, decoder and pose after its Adam step
    (fp32) and its loss with the free-space and SDF parts (fp64); ~2 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"embeddings": emb, "pose": pose6}
    arrays.update({"decoder." + k: v for k, v in dec.state_dict().items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "loss.npy"), np.array([st.loss, st.fs_loss, st.sdf_loss], np.float64))


def strong_scaling_block(nl, dev, rank, world, group, scan, ms, dec, steps, sync_all, timed, use_peer=False):
    """ONE scan, its rays split contiguously over the ranks (dist.shard_bounds), map / decoder / pose replicated, the three
    collectives of nerf-loam_b200/dist.py per step.  Also checks the parity gate of SURVEY 8(d): the all-reduced gradients of the
    sharded step equal those of an unsharded (1-rank) step over the same rays."""
    import torch.distributed as dist
    pts, cos, pose = scan
    h_dirs, h_gt, h_cos = host_rays(pts, cos)
    R = h_dirs.shape[0]
    lo, hi = nl.dist.shard_bounds(R, rank, world)
    dirs_all, gt_all, cos_all = h_dirs.to(dev), h_gt.to(dev), h_cos.to(dev)
    dirs, gt, cosv = dirs_all[lo:hi].contiguous(), gt_all[lo:hi].contiguous(), cos_all[lo:hi].contiguous()
    pose6 = nl.se3pose.OptimizablePose.from_matrix(torch.from_numpy(pose)).data.detach().reshape(1, 6).to(dev).contiguous()
    bufs = nl.engine.DecoderBuffers(dec, dev)
    Rl = hi - lo
    eng = nl.engine.SDFEngine(Rl, Rl * 20, dev)
    # ---- gradient equivalence (deterministic sampling, per-ray sampler tail: the reference's tail quirk depends on a ray's position
    #      in the batch, DESIGN.md deviation 6) ----
    kw = dict(n_frames=1, rng_seed=0, reference_compat=False, update_decoder=True, update_emb=True, update_pose=True, pose6=pose6)
    eng.rays_from_poses(pose6, dirs, None)
    eng.forward_backward(ms, bufs, Rl, CFG, gt, cosv, dir_local=dirs, ray_frame=None, group=group, **kw)
    torch.cuda.synchronize()
    g_sh = [eng.grad_emb.clone(), bufs.gradflat.clone(), eng.pose_grad.clone()]
    loss_sh = eng.read_stats().loss
    eng1 = nl.engine.SDFEngine(R, R * 20, dev)
    bufs1 = nl.engine.DecoderBuffers(dec, dev)
    eng1.rays_from_poses(pose6, dirs_all, None)
    eng1.forward_backward(ms, bufs1, R, CFG, gt_all, cos_all, dir_local=dirs_all, ray_frame=None, group=None, **kw)
    torch.cuda.synchronize()
    g_1 = [eng1.grad_emb, bufs1.gradflat, eng1.pose_grad]
    loss_1 = eng1.read_stats().loss
    rel = [float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) for a, b in zip(g_sh, g_1)]
    t = torch.tensor(rel + [abs(loss_sh - loss_1) / abs(loss_1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del eng1, bufs1
    torch.cuda.empty_cache()
    # ---- timing ----
    emb = ms.emb.clone()
    peer = pstats = None
    if use_peer:
        peer = nl.dist.PeerReduceAdam(group, dev, emb.shape[0], 1, lr=LR[0])
        peer.param.copy_(emb)
        emb = peer.param
        eng.adopt_gradflat(peer.grad, emb.shape[0], 1)
        pstats = nl.dist.PeerStats(group, dev)
    ms_s = nl.engine.MapState(ms.centres, ms.structure, ms.vox2row, emb, dev)
    opt = {"o": None}

    def step():
        eng.rays_from_poses(pose6, dirs, None)
        eng.forward_backward(ms_s, bufs, Rl, CFG, gt, cosv, dir_local=dirs, ray_frame=None, n_frames=1, rng_seed=12345, update_decoder=True,
                             update_emb=True, update_pose=True, pose6=pose6, group=group, defer_wgrad=eng.overlap_wgrad, peer=peer, peer_stats=pstats)
        if opt["o"] is None:
            opt["o"] = nl.engine.FusedAdam(([] if peer is not None else [dict(param=emb, grad=eng.grad_emb, lr=LR[0])]) +
                                           [dict(param=p.data.clone(), grad=g, lr=LR[1], side=True) for p, g in zip(bufs.params, bufs.grads)] +
                                           [dict(param=pose6[0], grad=eng.pose_grad[0], lr=LR[2])], ctl=lambda: eng.ctl)
        opt["o"].step(side_stream=eng.deferred_stream())
    eng.begin_call()
    for _ in range(10):
        step()
    ms_t = timed(step, steps, eng.join_side)
    n_loc = eng.read_stats().n_samples
    tt = torch.tensor([ms_t, float(n_loc)], dtype=torch.float64, device=dev)
    tm = tt.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ts = tt.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
    return {"scaling": "strong", "what": "ONE 82.7k-ray scan, rays split contiguously over the ranks (BASELINE.json config 5)", "rays_total": R,
            "samples_total": float(ts[1]), "ms_per_step": float(tm[0]) / steps, "value": float(ts[1]) * steps / (float(tm[0]) * 1e-3), "unit": "samples/s",
            "grad_equiv_max_rel": {"embedding": float(t[0]), "decoder": float(t[1]), "pose": float(t[2]), "loss": float(t[3]),
                                   "gate": 1e-5, "note": "max |g_sharded+allreduced - g_1rank| / max |g_1rank| over all ranks; deterministic noise, "
                                                         "reference_compat=False (per-ray sampler tail)"}}


# ======================================================================================================
# Baseline B (BASELINE.md section 3): the UNMODIFIED reference on the same B200 -- its eager PyTorch loop
# (oracle/_ref/src/variations/render_helpers.py, staged byte for byte) + its own CUDA extension (oracle/_ref/grid/grid_ref.so,
# compiled for sm_100a from the sources where they lie).  Baseline legs only; never on the product path.
# ======================================================================================================
class _TimedExt:
    """Proxy for the reference's `grid` extension that brackets its two live kernels with CUDA events."""

    def __init__(self, ext):
        self._ext, self.ev = ext, {"svo_intersect": [], "inverse_cdf_sampling": []}

    def _wrap(self, name):
        fn = getattr(self._ext, name)

        def call(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out = fn(*a); e1.record()
            self.ev[name].append((e0, e1))
            return out
        return call

    def __getattr__(self, name):
        return self._wrap(name) if name in self.ev else getattr(self._ext, name)

    def ms(self, name):
        torch.cuda.synchronize()
        return float(sum(a.elapsed_time(b) for a, b in self.ev[name]))


def _ref_frame(ref, index, pts, cos, pose, all_rays=False):
    # device-resident scan tensors: the reference indexes frame.rays_d with a CUDA mask (render_helpers.py:371-372), which torch >= 2
    # rejects for CPU tensors; this also turns its per-iteration uploads into no-ops (in the reference's favour)
    f = ref.LidarFrame(index, torch.from_numpy(pts).cuda(), torch.from_numpy(cos).cuda(),
                       ref.OptimizablePose(ref.OptimizablePose.from_matrix(torch.from_numpy(pose.copy())).data.detach().clone()), new_keyframe=True)
    if all_rays:    # the metric excludes host ray selection (SURVEY 8 d): every point is selected, the CPU Gumbel top-k is skipped
        f.sample_mask = torch.ones((f.num_point, 1), dtype=torch.bool, device="cuda")
        f.sample_rays = lambda *a, **k: None
    return f


def reference_gpu(nl, dev, steps, full_scan_pts, window_scans):
    """Times the reference's own bundle_adjust_frames / track_frame / kernels on this GPU.  full_scan_pts = (pts, cos, pose) of the
    headline scan; window_scans = list of scans of a 5-frame keyframe window (kitti.yaml: window_size 4 + current)."""
    from oracle import ref_harness as H
    if not H.available():
        return {"unavailable": "oracle/_ref (grid_ref.so + staged reference Python) not present on this box"}
    import copy
    ref = H.load()
    syn = nl.synthetic
    vs = CFG["voxel_size"]
    crit = ref.Criterion(H.args(CFG["max_depth"], CFG["truncation"], CFG["fs_weight"], CFG["sdf_weight"]))
    out = {"what": "unmodified reference (src/variations/render_helpers.py + voxel_helpers.py + grid CUDA extension built for sm_100a), "
                   "same B200, same synthetic scans; wall clock between torch.cuda.synchronize() (the reference syncs the host several "
                   "times per iteration itself)"}

    def build_map(scans):
        o = nl.svo.Octree(); o.init(256 * 256 * 4, 16, vs)          # bit-exact stand-in for the reference svo (tests/test_host_cpu.py)
        for pts, cos, pose in scans:
            o.insert(torch.from_numpy(syn.voxelize(pts, pose, vs)))
        v, c, f = o.get_centres_and_children()
        return H.reference_map_states(v, c, f, vs, init_std=0.01, seed=777, device=dev)

    def decoder():
        torch.manual_seed(777)
        return ref.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).to(dev)

    def wall(fn, n):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / n * 1e3

    # ---- (1) headline workload: one mapping iteration on ALL rays of the scan, decoder + embeddings + pose updated ----
    pts, cos, pose = full_scan_pts
    ms1 = build_map([full_scan_pts])
    dec1 = decoder()
    fr = _ref_frame(ref, 1, pts, cos, pose, all_rays=True)
    R = fr.num_point
    kw = dict(voxel_size=vs, step_size=CFG["step_size"], N_rays=R, truncation=CFG["truncation"], max_voxel_hit=20,
              max_distance=CFG["max_distance"], learning_rate=list(LR), update_pose=True, update_decoder=True)
    with H.pinned(ref, deterministic=False, stable_sort=False):
        # sample count of this workload from the reference's own renderer
        T = torch.from_numpy(pose).to(dev)
        P = torch.from_numpy(pts).to(dev)
        rd = ((P / (P.norm(dim=-1, keepdim=True) + 1e-8)) @ T[:3, :3].T)[None].contiguous()
        ro = T[:3, 3].reshape(1, 1, 3).expand_as(rd).contiguous()
        # (no torch.no_grad(): the reference's render_rays calls autograd.grad(sdf, xyz) itself, render_helpers.py:293-297)
        o1 = ref.orig["render_rays"](ro, rd, ms1, dec1, CFG["step_size"], vs, CFG["truncation"], 20, CFG["max_distance"], chunk_size=-1)
        M = int(o1["valid_mask"].sum())
        del o1
        run1 = lambda n: ref.orig["bundle_adjust_frames"]([fr], ms1["voxel_vertex_emb"], ms1, dec1, crit, num_iterations=n, **kw)
        run1(2)
        n_it = max(3, min(steps, 10))
        t_it = wall(lambda: run1(n_it), 1) / n_it
        # kernel-only time of the reference's two CUDA kernels inside one such iteration
        proxy = _TimedExt(ref.VH._ext)
        ref.VH._ext = proxy
        try:
            ref.orig["render_rays"](ro, rd, ms1, dec1, CFG["step_size"], vs, CFG["truncation"], 20, CFG["max_distance"], chunk_size=-1)
            k_int, k_smp = proxy.ms("svo_intersect"), proxy.ms("inverse_cdf_sampling")
        finally:
            ref.VH._ext = proxy._ext
    out["full_scan_iteration"] = {"rays": R, "samples": M, "ms_per_iter": t_it, "samples_per_s": M / (t_it * 1e-3), "iterations_timed": n_it,
                                  "note": "bundle_adjust_frames([frame], N_rays = all points), host ray selection skipped (metric definition)"}
    out["kernels"] = {"svo_intersect_ms": k_int, "inverse_cdf_sampling_ms": k_smp,
                      "note": "CUDA events around the reference's own kernel launches (intersect_gpu.cu:193-272, sample_gpu.cu:133-239) "
                              "for the full scan, inputs already materialised by its wrapper (octree copies not counted)"}
    del ms1, dec1
    torch.cuda.empty_cache()

    # ---- (2) the reference's real iteration size: 5 frames x 2048 rays, 25 iterations (configs/kitti/kitti.yaml:19-33) ----
    msw = build_map(window_scans)
    decw = decoder()
    frames = [_ref_frame(ref, i, *sc) for i, sc in enumerate(window_scans)]
    kww = dict(voxel_size=vs, step_size=CFG["step_size"], N_rays=2048, num_iterations=25, truncation=CFG["truncation"], max_voxel_hit=20,
               max_distance=CFG["max_distance"], learning_rate=list(LR), update_pose=True, update_decoder=True)
    with H.pinned(ref, deterministic=False, stable_sort=False):
        ba = lambda: ref.orig["bundle_adjust_frames"](frames, msw["voxel_vertex_emb"], msw, decw, crit, **kww)
        ba()
        t_ba = wall(ba, 2)
        # ---- (3) tracking: 25 iterations x 2048 rays against the same map ----
        ft = _ref_frame(ref, 5, *window_scans[-1])
        tk = lambda: ref.orig["track_frame"](copy.deepcopy(ft.pose), ft, msw, decw, crit, vs, N_rays=2048, step_size=0.2 * vs, num_iterations=25,
                                             truncation=CFG["truncation"], learning_rate=0.06, max_voxel_hit=20, max_distance=CFG["max_distance"],
                                             depth_variance=True)
        tk()
        t_tk = wall(tk, 3)
    out["bundle_adjust_frames_5x2048x25"] = {"ms_per_call": t_ba, "frames": len(frames), "rays_per_frame": 2048, "iterations": 25,
                                             "includes": "the reference's per-iteration CPU ray selection (frame.sample_rays)"}
    out["track_frame_2048x25"] = {"ms_per_scan": t_tk}
    return out


def ours_real_size(nl, dev, window_scans, ms, dec):
    """The drop-in bundle_adjust_frames / track_frame at the reference's real iteration size, same scans as reference_gpu (2)/(3)."""
    from types import SimpleNamespace
    import copy
    crit = nl.criterion.Criterion(SimpleNamespace(criteria={"eiko_weight": 0.1, "sdf_weight": CFG["sdf_weight"], "fs_weight": CFG["fs_weight"],
                                                           "sdf_truncation": CFG["truncation"]}, data_specs={"max_depth": CFG["max_depth"]}))
    vs = CFG["voxel_size"]
    frames = []
    for i, (pts, cos, pose) in enumerate(window_scans):
        frames.append(nl.frame.LidarFrame(i, torch.from_numpy(pts), torch.from_numpy(cos),
                                          nl.se3pose.OptimizablePose.from_matrix(torch.from_numpy(pose.copy())), new_keyframe=True))
    res = {}
    for name, mode, graph in (("host_selection", "host", False), ("device_selection", "device", False), ("cuda_graph", "device", True)):
        def ba():
            nl.render_helpers.bundle_adjust_frames(frames, ms.emb, ms, dec, crit, vs, CFG["step_size"], N_rays=2048, num_iterations=25,
                                                   truncation=CFG["truncation"], max_voxel_hit=20, max_distance=CFG["max_distance"],
                                                   learning_rate=list(LR), update_pose=True, update_decoder=True, ray_selection=mode, cuda_graph=graph)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        ba(); torch.cuda.synchronize()
        res["ms_first_call_%s" % name] = (time.perf_counter() - t0) * 1e3          # includes the graph capture where there is one
        t0 = time.perf_counter()
        for _ in range(3):
            ba()
        torch.cuda.synchronize()
        res["ms_per_call_%s" % name] = (time.perf_counter() - t0) / 3 * 1e3
    res.update(frames=len(frames), rays_per_frame=2048, iterations=25)
    return res


# BASELINE.json configs 1-3 at their real iteration sizes (configs/maicity/maicity.yaml, configs/kitti/kitti.yaml, configs/ncd/ncd.yaml):
# window of keyframes x 2048 rays through the drop-in bundle_adjust_frames / track_frame on a map grown incrementally, + mesh extraction
REAL_CONFIGS = {
    "config1_maicity": dict(voxel=0.2, map_step=0.5, map_it=20, track_step=0.2, track_it=20, track_lr=0.06, window=5, max_depth=50.0, min_depth=1.5, lr=(0.01, 0.005, 0.001)),
    "config2_kitti": dict(voxel=0.3, map_step=0.5, map_it=25, track_step=0.2, track_it=25, track_lr=0.06, window=5, max_depth=40.0, min_depth=5.0, lr=(0.01, 0.005, 0.001)),
    "config3_newer_college": dict(voxel=0.2, map_step=0.2, map_it=15, track_step=0.1, track_it=30, track_lr=0.04, window=6, max_depth=40.0, min_depth=1.0, lr=(0.002, 0.005, 0.001)),
}


def configs_real_size(nl, dev):
    from types import SimpleNamespace
    syn = nl.synthetic
    out = {}
    for name, c in REAL_CONFIGS.items():
        vs = c["voxel"]
        crit = nl.criterion.Criterion(SimpleNamespace(criteria={"eiko_weight": 0.1, "sdf_weight": 10000.0, "fs_weight": 1.0, "sdf_truncation": 0.3},
                                                      data_specs={"max_depth": c["max_depth"]}))
        scans = [syn.make_scan(seed=900 + i, sensor_xyz=(1.0 * i, 0.0, 0.0), min_depth=c["min_depth"], max_depth=c["max_depth"]) for i in range(c["window"])]
        mu = nl.mapping.MapUpdater(vs, init_std=0.01, seed=777, device=dev)
        t_upd = []
        for pts, cos, pose in scans:
            vox = torch.from_numpy(syn.voxelize(pts, pose, vs))
            torch.cuda.synchronize(); t0 = time.perf_counter()
            ms = mu.insert_voxels(vox)
            torch.cuda.synchronize(); t_upd.append((time.perf_counter() - t0) * 1e3)
        torch.manual_seed(777)
        dec = nl.lidar.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).to(dev)
        frames = [nl.frame.LidarFrame(i, torch.from_numpy(p), torch.from_numpy(cs), nl.se3pose.OptimizablePose.from_matrix(torch.from_numpy(T.copy())), new_keyframe=True)
                  for i, (p, cs, T) in enumerate(scans)]

        def ba():
            nl.render_helpers.bundle_adjust_frames(frames, mu.embeddings, ms, dec, crit, vs, c["map_step"] * vs, N_rays=2048, num_iterations=c["map_it"],
                                                   truncation=0.3, max_voxel_hit=20, max_distance=c["max_depth"], learning_rate=list(c["lr"]))

        def tk():
            return nl.render_helpers.track_frame(frames[-1].pose, frames[-1], ms, dec, crit, vs, N_rays=2048, step_size=c["track_step"] * vs,
                                                 num_iterations=c["track_it"], truncation=0.3, learning_rate=c["track_lr"], max_voxel_hit=20,
                                                 max_distance=c["max_depth"])
        res = {}
        for key, fn, n in (("bundle_adjust_frames_ms", ba, 3), ("track_frame_ms", tk, 5)):
            fn(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
            res[key] = (time.perf_counter() - t0) / n * 1e3
        nl.mesh.extract_mesh(dec, ms, vs, res=8); torch.cuda.synchronize()
        t0 = time.perf_counter()
        v, f = nl.mesh.extract_mesh(dec, ms, vs, res=8)
        torch.cuda.synchronize()
        res.update(extract_mesh_res8_ms=(time.perf_counter() - t0) * 1e3, mesh_vertices=int(v.shape[0]), mesh_triangles=int(f.shape[0]),
                   map_update_ms=[round(x, 2) for x in t_upd], octree_nodes=ms.n_nodes, last_update_dirty_rows=mu.last_update.get("dirty_rows"),
                   frames=len(frames), mapping_iterations=c["map_it"], tracking_iterations=c["track_it"], rays_per_frame=2048)
        out[name] = res
        del mu, ms, dec, frames
        torch.cuda.empty_cache()
    out["note"] = ("default drop-in paths: device-side ray selection, captured CUDA graph on the MapUpdater's stable buffers; wall clock per call; "
                   "map_update_ms = incremental octree insert + dirty-row export + device patch per scan; synthetic 64x1563-beam scans 1 m apart")
    return out


def cpu_baseline(n_rays=4096, iters=3, threads=None):
    """The oracle port of the reference path (oracle/: C traversal + sampler, torch fp32 chain, autograd,
    torch.optim.Adam) timed on this box's host cores on a bounded sample of the same workload."""
    from oracle import chain as OC
    from oracle import kernels as OK
    import importlib
    syn = importlib.import_module("nerf-loam_b200.synthetic")
    if threads is None:
        threads = int(os.environ.get("NL_CPU_THREADS", 0)) or min(os.cpu_count(), 32)   # eager PyTorch stops scaling (and then
    torch.set_num_threads(threads)                                                      # regresses) beyond a few dozen threads
    pts, cos, pose = syn.make_scan(seed=777)
    o = OK.Octree(); o.init(256 * 256 * 4, 16, CFG["voxel_size"])
    o.insert(syn.voxelize(pts, pose, CFG["voxel_size"]))
    voxels, children, features = o.get_centres_and_children()
    centres, structure, vertex = OK.map_arrays(voxels, children, features, CFG["voxel_size"])
    flat = vertex.reshape(-1); used = flat[flat >= 0]
    uniq, first = np.unique(used, return_index=True)
    v2r = np.full(vertex.shape[0], -1, np.int64); v2r[uniq[np.argsort(first)]] = np.arange(len(uniq))
    map_np = {"centres": centres, "structure": structure, "vertex_rows": np.where(vertex >= 0, v2r[np.clip(vertex, 0, None)], -1)}
    g = torch.Generator().manual_seed(777)
    emb = (torch.randn(len(uniq), 16, generator=g) * 0.01).to(torch.bfloat16).requires_grad_()
    torch.manual_seed(777)
    dec = OC.Decoder(depth=2, width=256, in_dim=16)
    pose6 = torch.nn.Parameter(OC.pose_from_matrix(torch.from_numpy(pose)))
    opt = torch.optim.Adam([{"params": [emb], "lr": LR[0]}, {"params": list(dec.parameters()), "lr": LR[1]}, {"params": [pose6], "lr": LR[2]}])
    sel = np.random.default_rng(0).choice(pts.shape[0], n_rays, replace=False); sel.sort()
    P = torch.from_numpy(pts[sel]); C_ = torch.from_numpy(cos[sel])
    frame = dict(pose=pose6, dirs=P / (P.norm(dim=-1, keepdim=True) + 1e-8), points=P, cos=C_)
    cfg = dict(CFG)
    times, nsamp = [], 0
    for it in range(iters + 1):
        t0 = time.perf_counter()
        loss, out = OC.mapping_iteration([frame], map_np, emb, dec, cfg, deterministic=True)
        opt.zero_grad(); loss.backward(); opt.step()
        dt = time.perf_counter() - t0
        nsamp = int(out["valid_mask"].sum())
        if it > 0:
            times.append(dt)
    return {"value": nsamp / float(np.median(times)), "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": f"{n_rays} rays of the same scan ({nsamp} samples) per iteration, median of {iters} after 1 warm-up; "
                      "oracle port: C traversal/sampler + PyTorch fp32 CPU chain + autograd + torch.optim.Adam",
            "ms_per_iter": float(np.median(times)) * 1e3}


def best_cpu_baseline(n_rays, iters):
    """Pick the thread count at which the host path is fastest (a fair baseline: eager PyTorch on 128 threads is
    ~100x slower than on 16) and report that run; `cores` is the thread count actually used."""
    best = None
    for th in sorted({min(os.cpu_count(), t) for t in (8, 16, 32)}):
        cb = cpu_baseline(n_rays=n_rays, iters=1, threads=th)
        if best is None or cb["value"] > best["value"]:
            best = cb
    full = cpu_baseline(n_rays=n_rays, iters=iters, threads=best["cores"])
    full["sample"] += f"; thread count chosen as the fastest of 8/16/32 on a {os.cpu_count()}-CPU host"
    return full


def run_reference(args):
    """Reference arm.  The reference's stock code path for this metric is a GPU path (eager PyTorch + its own CUDA extension), so when
    the staged reference (oracle/_ref: grid_ref.so built for sm_100a + its unmodified Python) and a GPU are present the line's value
    is THAT -- Baseline B of BASELINE.md, the same workload, same B200 -- and the CPU port of the path (Baseline A, host cores) is
    reported beside it in `cpu_baseline`.  Without them the CPU port is the value."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    t0 = time.perf_counter()
    n_rays = 8192
    probe = best_cpu_baseline(n_rays=2048, iters=1)
    cb = cpu_baseline(n_rays=n_rays, iters=max(1, min(args.steps, 10)), threads=probe["cores"])
    gpu = None
    try:
        from oracle import ref_harness as H
        if torch.cuda.is_available() and H.available():
            import nerfloam_b200 as nl          # synthetic scan generator + the (bit-exact) octree builder only
            dev = torch.device("cuda", 0)
            torch.cuda.set_device(dev)
            gpu = reference_gpu_headline(nl, dev, args.steps, args.warmup)
    except Exception as exc:
        gpu = {"error": repr(exc)}
    out = {"impl": "reference", "metric": "neural-SDF samples/sec per mapping iter", "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "gpu_launches": 0, "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}}
    if gpu and "value" in gpu:
        out.update(value=gpu["value"], ms_per_step=gpu["ms_per_step"],
                   config={"workload": WORKLOAD, "rays_per_gpu": gpu["rays"], "samples_per_gpu_step": gpu["samples"],
                           "note": "UNMODIFIED reference (src/variations/render_helpers.py::bundle_adjust_frames + voxel_helpers.py + grid CUDA extension "
                                   "compiled for sm_100a) on this box's GPU 0: one mapping iteration on all rays of the same scan per step, decoder + "
                                   "embeddings + pose updated by torch.optim.Adam; host ray selection skipped (metric definition); wall clock between "
                                   "torch.cuda.synchronize() calls.  cpu_baseline = the oracle's CPU port of the same path on host cores"},
                   e2e={"value": gpu["value"], "unit": "samples/s", "h2d_bytes_per_step": gpu["h2d_bytes_per_step"], "d2h_bytes_per_step": 0,
                        "note": "scan tensors device-resident (see _ref_frame): the reference's own per-iteration uploads are no-ops here"},
                   reference_kind="reference-gpu")
    else:
        out.update(value=cb["value"], ms_per_step=cb["ms_per_iter"],
                   config={"workload": WORKLOAD, "note": f"reference algorithm on host cores (oracle port); each step = a bounded sample of {n_rays} rays",
                           "gpu_reference": gpu},
                   e2e={"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, reference_kind="cpu-port")
    out["wall_s"] = time.perf_counter() - t0
    print(json.dumps(out))


def reference_gpu_headline(nl, dev, steps, warmup):
    """The reference's own bundle_adjust_frames on ALL rays of the headline scan: `warmup` + `steps` iterations, wall clock."""
    from oracle import ref_harness as H
    ref = H.load()
    syn = nl.synthetic
    vs = CFG["voxel_size"]
    pts, cos, pose = syn.make_scan(seed=777)
    o = nl.svo.Octree(); o.init(256 * 256 * 4, 16, vs)
    o.insert(torch.from_numpy(syn.voxelize(pts, pose, vs)))
    v, c, f = o.get_centres_and_children()
    ms1 = H.reference_map_states(v, c, f, vs, init_std=0.01, seed=777, device=dev)
    torch.manual_seed(777)
    dec1 = ref.Decoder(depth=2, width=256, in_dim=16, skips=[], embedder="none", multires=0).to(dev)
    crit = ref.Criterion(H.args(CFG["max_depth"], CFG["truncation"], CFG["fs_weight"], CFG["sdf_weight"]))
    fr = _ref_frame(ref, 1, pts, cos, pose, all_rays=True)
    R = fr.num_point
    kw = dict(voxel_size=vs, step_size=CFG["step_size"], N_rays=R, truncation=CFG["truncation"], max_voxel_hit=20,
              max_distance=CFG["max_distance"], learning_rate=list(LR), update_pose=True, update_decoder=True)
    with H.pinned(ref, deterministic=False, stable_sort=False):
        T = torch.from_numpy(pose).to(dev)
        P = torch.from_numpy(pts).to(dev)
        rd = ((P / (P.norm(dim=-1, keepdim=True) + 1e-8)) @ T[:3, :3].T)[None].contiguous()
        ro = T[:3, 3].reshape(1, 1, 3).expand_as(rd).contiguous()
        # (no torch.no_grad(): the reference's render_rays calls autograd.grad(sdf, xyz) itself, render_helpers.py:293-297)
        o1 = ref.orig["render_rays"](ro, rd, ms1, dec1, CFG["step_size"], vs, CFG["truncation"], 20, CFG["max_distance"], chunk_size=-1)
        M = int(o1["valid_mask"].sum())
        del o1
        run = lambda n: ref.orig["bundle_adjust_frames"]([fr], ms1["voxel_vertex_emb"], ms1, dec1, crit, num_iterations=n, **kw)
        run(max(1, warmup))
        torch.cuda.synchronize(); t0 = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    return {"value": M * steps / dt, "ms_per_step": dt / steps * 1e3, "rays": R, "samples": M, "h2d_bytes_per_step": 0}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    a = ap.parse_args()
    # stdout carries exactly one JSON line: while the benchmark runs, file descriptor 1 points at stderr, so that library
    # banners written with printf (NCCL prints its version there) cannot get in front of it
    sys.stdout.flush()
    _saved_stdout = os.dup(1)
    os.dup2(2, 1)
    _real_print = print

    def print(*args, **kw):   # noqa: A001  (the two result prints below go to the real stdout)
        sys.stdout.flush()
        os.dup2(_saved_stdout, 1)
        _real_print(*args, **kw)
        sys.stdout.flush()
        os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device for --impl ours (there is no CPU fallback)")
        run_ours(a)
