"""GPU parity tests of the individual C-ABI ops against the oracle, the golden vectors produced by the
executed reference, and the outputs of the compiled unmodified reference kernels recorded on a B200
(tests/golden/reference_gpu.npz, tests/golden/make_golden_gpu.py)."""
import numpy as np
import pytest
import torch

from util import bf16_from_bits, golden, product_map, load_decoder

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nl():
    import nerfloam_b200 as nl
    assert torch.cuda.is_available()
    return nl


@pytest.fixture(scope="module")
def scene(nl):
    z = golden("render.npz")
    m = product_map(z["vox"], float(z["voxel_size"]), z["id2emb"], z["emb_bf16"])
    return z, m


def canon_ties(idx, mn, mx):
    """Order hits with bit-identical min_depth canonically (the tie order is unspecified in the reference)."""
    key = np.lexsort((idx, mn), axis=-1) if False else None
    out_i, out_a, out_b = idx.copy(), mn.copy(), mx.copy()
    for r in range(idx.shape[0]):
        o = np.lexsort((idx[r], mn[r]))
        out_i[r], out_a[r], out_b[r] = idx[r][o], mn[r][o], mx[r][o]
    return out_i, out_a, out_b


def test_svo_intersect_vs_oracle_and_reference(nl, scene):
    from oracle import kernels as OK
    z, m = scene
    vs = float(z["voxel_size"])
    ro = torch.from_numpy(z["rays_o"]).cuda()[None].contiguous()
    rd = torch.from_numpy(z["rays_d"]).cuda()[None].contiguous()
    pts = m["centres"].cuda()[None].contiguous()
    ch = m["structure"].cuda()[None].contiguous()
    idx, mn, mx = nl.grid.svo_intersect(ro, rd, pts, ch, vs, 20)
    oi, omn, omx = OK.svo_intersect(z["rays_o"], z["rays_d"], m["centres"].numpy(), m["structure"].numpy(), vs, 20)
    assert np.array_equal(idx[0].cpu().numpy(), oi)                     # voxel ids: bit-exact, DFS order
    np.testing.assert_allclose(mn[0].cpu().numpy(), omn, rtol=2e-6, atol=1e-6)   # __fdividef vs 1.0f/x
    np.testing.assert_allclose(mx[0].cpu().numpy(), omx, rtol=2e-6, atol=1e-6)
    # the real reference kernel on a B200, called the way its wrapper calls it (rays batched, octree replicated per batch)
    r = golden("reference_gpu.npz")
    mi, mmn, mmx = nl.grid.svo_intersect(*intersect_batched(ro, rd, pts, ch), vs, 20)
    rows = torch.from_numpy(r["isect_rows"]).long()
    for got, want in ((mi, r["isect_idx"]), (mmn, r["isect_min"]), (mmx, r["isect_max"])):
        assert torch.equal(got.reshape(-1, 20)[rows].cpu(), torch.from_numpy(want))      # bit-exact incl. depths


def intersect_batched(ro, rd, pts, ch, G=4):
    """svo_intersect's inputs as the reference's wrapper lays them out: rays in G batches, the octree replicated per batch."""
    K = ro.shape[1] // G
    rep = lambda a: a.expand(G, -1, -1).contiguous()
    return ro[:, :G * K].reshape(G, K, 3).contiguous(), rd[:, :G * K].reshape(G, K, 3).contiguous(), rep(pts), rep(ch)


def inverse_cdf_inputs(z):
    """inverse_cdf_sampling's inputs for the hit rays of render.npz: [Gb, H/Gb, P] hits padded by repeating the first ray, seeded
    noise, probabilities and step counts as the reference's ray_sample computes them."""
    from oracle import kernels as OK
    hits = z["hits"]
    P = z["hit_idx"].shape[1]
    idx = z["hit_idx"][hits]; mn = z["hit_min"][hits]; mx = z["hit_max"][hits]
    d = (mx - mn).astype(np.float32); d[idx == -1] = 0
    tot = OK.seq_sum(d)
    probs = (d / tot[:, None]).astype(np.float32)
    steps = (tot / np.float32(z["step"])).astype(np.float32)
    N = idx.shape[0]
    Gb = 200
    H = int(np.ceil(N / Gb)) * Gb
    pad = lambda a: np.concatenate([a, np.broadcast_to(a[:1], (H - N,) + a.shape[1:])], 0)
    I, A, B, PR, ST = [pad(a) for a in (idx, mn, mx, probs, steps)]
    S = int(np.ceil(ST).max()) + P
    rng = np.random.default_rng(0)
    noise = rng.uniform(0.001, 0.999, size=(Gb, H // Gb, S)).astype(np.float32)
    shp = (Gb, H // Gb, P)
    t = lambda a, s: torch.from_numpy(np.ascontiguousarray(a.reshape(s))).cuda()
    return t(I, shp), t(A, shp), t(B, shp), torch.from_numpy(noise).cuda(), t(PR, shp), t(ST, (Gb, H // Gb))


def test_inverse_cdf_sampling_vs_oracle_and_reference(nl, scene):
    from oracle import kernels as OK
    z, m = scene
    args = inverse_cdf_inputs(z)
    Gb, Hb, P = args[0].shape
    S = args[3].shape[-1]
    si, sd, sl = nl.grid.inverse_cdf_sampling(*args, -1.0)
    oi = np.empty((Gb, Hb, S), np.int32); od = np.empty_like(oi, dtype=np.float32); ol = np.empty_like(od)
    a = [np.ascontiguousarray(x.cpu().numpy()) for x in args]
    OK.lib().nlo_inverse_cdf_sampling(Gb, Hb, P, S, -1.0, OK._p(a[0]), OK._p(a[1]), OK._p(a[2]), OK._p(a[3]), OK._p(a[4]),
                                      OK._p(a[5]), OK._p(oi), OK._p(od), OK._p(ol))
    assert np.array_equal(si.cpu().numpy(), oi)
    assert np.array_equal(sd.cpu().numpy(), od) and np.array_equal(sl.cpu().numpy(), ol)   # same fp ops incl. the FMA
    r = golden("reference_gpu.npz")                                    # the compiled reference kernel on a B200
    rows = torch.from_numpy(r["icdf_rows"]).long()
    for got, want in ((si, r["icdf_idx"]), (sd, r["icdf_depth"]), (sl, r["icdf_dist"])):
        assert torch.equal(got.reshape(Gb * Hb, S)[rows].cpu(), torch.from_numpy(want))


def test_reference_grid_pins_the_oracle(nl, scene):
    """The oracle's C restatement of the two CUDA kernels against the compiled reference itself (its outputs recorded on a B200
    for the rays of tests/golden/reference_gpu.npz)."""
    from oracle import kernels as OK
    z, m = scene
    vs = float(z["voxel_size"])
    r = golden("reference_gpu.npz")
    rows = r["isect_rows"]
    oi, omn, omx = OK.svo_intersect(z["rays_o"][rows], z["rays_d"][rows], m["centres"].numpy(), m["structure"].numpy(), vs, 20)
    assert np.array_equal(r["isect_idx"], oi)
    np.testing.assert_allclose(r["isect_min"], omn, rtol=2e-6, atol=1e-6)


@pytest.mark.parametrize("width", [256, 32])
def test_gather_and_mlp_vs_reference_golden(nl, width):
    """get_embeddings + Decoder forward/backward (reference Python, executed on CPU) vs the CUDA kernels."""
    z = golden("chain.npz")
    M = z["xyz"].shape[0]
    vs = float(z["voxel_size"])
    dev = "cuda"
    # every sample gets its own voxel with its own 8 rows: table [M*8,16], vox2row[m] = 8m..8m+7
    emb = bf16_from_bits(z["feats_bf16"]).reshape(M * 8, 16).to(dev).contiguous()
    vox = torch.arange(M, dtype=torch.int32, device=dev)
    vox2row = torch.arange(M * 8, dtype=torch.int32, device=dev).reshape(M, 8).contiguous()
    centres = torch.from_numpy(z["centre"]).to(dev).contiguous()
    xyz = torch.from_numpy(z["xyz"]).to(dev).contiguous()
    feats = torch.empty((M, 16), dtype=torch.float32, device=dev)
    lib, cap = nl._capi.lib(), nl._capi
    cap.check(lib.nl_gather_trilinear_fwd(M, None, cap.ptr(xyz), cap.ptr(vox), cap.ptr(centres), cap.ptr(vox2row), cap.ptr(emb), vs,
                                          cap.ptr(feats), cap.stream_ptr()))
    np.testing.assert_allclose(feats.cpu().numpy(), z[f"w{width}_emb"], atol=1e-7, rtol=1e-6)

    dec = load_decoder(z, f"w{width}_p_", dev, width)
    x = feats.clone().requires_grad_()
    sdf = dec(x)["sdf"]
    np.testing.assert_allclose(sdf.detach().cpu().numpy(), z[f"w{width}_sdf"], atol=1e-5)      # north-star tolerance
    gout = torch.from_numpy(z[f"w{width}_gout"]).to(dev)
    (sdf * gout).sum().backward()
    for k, p in dec.state_dict(keep_vars=True).items():
        ref = z[f"w{width}_g_{k}"]
        np.testing.assert_allclose(p.grad.cpu().numpy(), ref, atol=1e-4 * max(1.0, np.abs(ref).max()), rtol=1e-4)
    # gather backward: d feats -> rows (bf16-rounded like autograd) and d xyz
    grad_emb = torch.zeros((M * 8, 16), dtype=torch.float32, device=dev)
    dxyz = torch.empty((M, 3), dtype=torch.float32, device=dev)
    dfe = x.grad.contiguous()
    cap.check(lib.nl_gather_trilinear_bwd(M, None, cap.ptr(xyz), cap.ptr(vox), cap.ptr(centres), cap.ptr(vox2row), cap.ptr(emb), vs,
                                          cap.ptr(dfe), 1, cap.ptr(grad_emb), cap.ptr(dxyz), None, None, None, None, 0, None,
                                          cap.stream_ptr()))
    ref_df = z[f"w{width}_dfeats"].reshape(M * 8, 16)
    got = grad_emb.cpu().numpy()
    # bf16 rounding of each contribution: equal up to one bf16 ulp where the fp32 product sat on a rounding boundary
    assert np.mean(np.abs(got - ref_df) > 1e-2 * np.abs(ref_df) + 1e-9) < 2e-3
    ref_dx = z[f"w{width}_dxyz"]
    np.testing.assert_allclose(dxyz.cpu().numpy(), ref_dx, atol=2e-4 * np.abs(ref_dx).max(), rtol=1e-3)


def test_pose_kernels_vs_reference_golden(nl):
    z = golden("pose.npz")
    dev = "cuda"
    lib, cap = nl._capi.lib(), nl._capi
    datas = torch.from_numpy(np.concatenate([z["data"][None], z["datas"]])).float().to(dev).contiguous()
    F = datas.shape[0]
    Rt = torch.empty((F, 12), dtype=torch.float32, device=dev)
    cap.check(lib.nl_pose_matrices(F, cap.ptr(datas), cap.ptr(Rt), cap.stream_ptr()))
    Rk = Rt[:, :9].reshape(F, 3, 3).cpu().numpy()
    np.testing.assert_allclose(Rk[0], z["R"], atol=2e-6)
    np.testing.assert_allclose(Rk[1:], z["Rs"], atol=2e-6)
    np.testing.assert_allclose(Rt[:, 9:].cpu().numpy(), datas[:, :3].cpu().numpy())
    # Jacobian: d (sum R*G) / d w  via acc = (dL/dt = 0, dL/dR = G)
    acc = torch.zeros((F, 12), dtype=torch.float32, device=dev)
    acc[:, 3:] = torch.from_numpy(z["G"]).reshape(1, 9).to(dev)
    acc[0, :3] = torch.from_numpy(z["gt"]).to(dev)
    g6 = torch.empty((F, 6), dtype=torch.float32, device=dev)
    cap.check(lib.nl_pose_grad(F, cap.ptr(datas), cap.ptr(acc), cap.ptr(g6), cap.stream_ptr()))
    np.testing.assert_allclose(g6[0].cpu().numpy(), z["grad"], atol=2e-5, rtol=1e-4)
    np.testing.assert_allclose(g6[1:, 3:].cpu().numpy(), z["grads"][:, 3:], atol=5e-5, rtol=2e-4)
    # the reference's own self-check (se3pose.py:95-105): from_matrix -> matrix round trip
    P = nl.se3pose.OptimizablePose.from_matrix(torch.from_numpy(z["before"]))
    np.testing.assert_allclose(P.matrix().detach().numpy()[:3, 3], z["before"][:3, 3], atol=1e-6)
    np.testing.assert_allclose(P.data.detach().numpy(), z["data"], atol=1e-6)


def test_fused_pose_launches_equal_the_separate_kernels_bit_for_bit(nl):
    """nl_rays_from_pose6 == nl_pose_matrices + nl_rays_from_poses, and nl_pose_step == nl_pose_grad + nl_adam_f32_ctl per selected
    pose + nl_loss_finalize + the two seed advances (what a captured iteration used to launch one by one)."""
    cap, lib = nl._capi, nl._capi.lib()
    dev = torch.device("cuda")
    torch.manual_seed(3)
    F, R = 5, 3001
    pose6 = (torch.randn(F, 6, device=dev) * torch.tensor([2, 2, 2, 0.3, 0.3, 0.3], device=dev)).contiguous()
    pose6[2, 3:] = 0                                                   # theta = 0 row (Taylor at 0, zero-angle derivative)
    dirs = torch.nn.functional.normalize(torch.randn(R, 3, device=dev), dim=-1).contiguous()
    fid = torch.randint(0, F, (R,), device=dev, dtype=torch.int32)
    st = cap.stream_ptr()
    Rt_a, Rt_b = torch.empty(F, 12, device=dev), torch.empty(F, 12, device=dev)
    o_a, d_a, o_b, d_b = (torch.empty(R, 3, device=dev) for _ in range(4))
    cap.check(lib.nl_pose_matrices(F, cap.ptr(pose6), cap.ptr(Rt_a), st))
    cap.check(lib.nl_rays_from_poses(R, cap.ptr(dirs), cap.ptr(fid), cap.ptr(Rt_a), cap.ptr(o_a), cap.ptr(d_a), st))
    cap.check(lib.nl_rays_from_pose6(R, F, cap.ptr(dirs), cap.ptr(fid), cap.ptr(pose6), cap.ptr(Rt_b), cap.ptr(o_b), cap.ptr(d_b), st))
    assert torch.equal(Rt_a, Rt_b) and torch.equal(o_a, o_b) and torch.equal(d_a, d_b)
    cap.check(lib.nl_rays_from_pose6(R, 1, cap.ptr(dirs), None, cap.ptr(pose6), None, cap.ptr(o_b), cap.ptr(d_b), st))     # tracking: one pose, no frame ids
    cap.check(lib.nl_rays_from_poses(R, cap.ptr(dirs), None, cap.ptr(Rt_a), cap.ptr(o_a), cap.ptr(d_a), st))
    assert torch.equal(o_a, o_b) and torch.equal(d_a, d_b)

    acc = torch.randn(F, 12, device=dev).contiguous()
    mask = 0b11010
    for skip, step in ((0, 1), (0, 7), (1, 7)):
        ctl = torch.zeros(cap.CTL_WORDS, dtype=torch.int32, device=dev)
        ctl[cap.CTL_ADAM_STEP], ctl[cap.CTL_SKIP_NOW] = step, skip
        stats = torch.zeros(nl.engine.STATS_BYTES, dtype=torch.uint8, device=dev)
        stats.view(torch.int32)[0], stats.view(torch.int32)[2] = 1000, 37
        stats.view(torch.float64)[16], stats.view(torch.float64)[17] = 123.456, 7.89
        f32 = stats.view(torch.float32)
        f32[26], f32[27], f32[30], f32[31] = 0.3, 0.7, 11.0, 5.0
        m0, v0 = torch.rand(F, 6, device=dev) * 1e-2, torch.rand(F, 6, device=dev) * 1e-4
        seeds0 = torch.tensor([2 ** 31 - 5, 12345], dtype=torch.int32, device=dev)
        # separate kernels
        pa, ma, va, sa, ga = pose6.clone(), m0.clone(), v0.clone(), stats.clone(), torch.empty(F, 6, device=dev)
        cap.check(lib.nl_pose_grad(F, cap.ptr(pa), cap.ptr(acc), cap.ptr(ga), st))
        cap.check(lib.nl_loss_finalize(cap.ptr(sa), 1.5, 1000.0, st))
        for f in range(F):
            if (mask >> f) & 1:
                cap.check(lib.nl_adam_f32_ctl(6, cap.ptr(pa[f]), cap.ptr(ga[f]), cap.ptr(ma[f]), cap.ptr(va[f]), 1e-3, 0.9, 0.999, 1e-8, cap.ptr(ctl), st))
        seeds_a = seeds0.clone()
        seeds_a[0:1].add_(0x632BE5); seeds_a[1:2].add_(0x3779B1)
        # one launch
        pb, mb, vb, sb, gb, seeds_b = pose6.clone(), m0.clone(), v0.clone(), stats.clone(), torch.empty(F, 6, device=dev), seeds0.clone()
        cap.check(lib.nl_pose_step(F, cap.ptr(pb), cap.ptr(acc), cap.ptr(gb), mask, cap.ptr(mb), cap.ptr(vb), 1e-3, 0.9, 0.999, 1e-8, cap.ptr(ctl),
                                   cap.ptr(sb), 1.5, 1000.0, cap.ptr(seeds_b[0:1]), 0x632BE5, cap.ptr(seeds_b[1:2]), 0x3779B1, st))
        torch.cuda.synchronize()
        assert torch.equal(ga, gb) and torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), (skip, step)
        assert torch.equal(sa, sb) and torch.equal(seeds_a, seeds_b)
        assert (not skip) == (not torch.equal(pb, pose6)) and torch.equal(pb[0], pose6[0]) and torch.equal(pb[2], pose6[2])   # rows 0 and 2 are not selected
        assert float(sb.view(torch.float32)[36]) != 0.0


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_fused_adam_vs_torch(nl, dtype):
    torch.manual_seed(0)
    dev = "cuda"
    n = 4096 * 16 + 7
    p0 = torch.randn(n, device=dev) * 0.05
    if dtype == "bf16":
        p0 = p0.to(torch.bfloat16)
    p_ref = p0.clone().requires_grad_()
    p_my = p0.clone()
    opt_ref = torch.optim.Adam([p_ref], lr=0.01)
    g32 = torch.zeros(n, dtype=torch.float32, device=dev)
    opt_my = nl.engine.FusedAdam([dict(param=p_my, grad=g32, lr=0.01)])
    for step in range(4):
        g = torch.randn(n, device=dev) * (10.0 ** (-step))
        if step == 2:
            g[::3] = 0
        p_ref.grad = g.to(p_ref.dtype)
        g32.copy_(g)
        opt_ref.step()
        opt_my.step()
        a, b = p_my.float().cpu().numpy(), p_ref.detach().float().cpu().numpy()
        if dtype == "f32":
            np.testing.assert_allclose(a, b, rtol=2e-6, atol=1e-8)
        else:   # same rounding points: identical up to rare 1-ulp flips from reciprocal-vs-division inside torch
            assert np.mean(a != b) < 2e-2
            np.testing.assert_allclose(a, b, rtol=1e-2, atol=1e-4)


def test_fused_adam_side_stream_is_ordered_behind_the_moments_zero_fill(nl):
    """bundle_adjust_frames updates the decoder on the engine's side stream (engine.SDFEngine.forward_backward, defer_wgrad).  The
    optimiser's moments are zero-filled on the MAIN stream when it is constructed, after the side stream forked: without an explicit
    dependency the first side-stream step may read whatever the recycled blocks held (NaN moments -> NaN decoder after a few calls of a
    loop that never synchronises).  Made deterministic here: the recycled blocks hold NaN and the main stream is stalled."""
    dev = torch.device("cuda")
    n = 64 * 1024
    p = torch.ones(n, device=dev)
    g = torch.full((n,), 0.5, device=dev)
    side = torch.cuda.Stream(device=dev)
    poison = [torch.full((n,), float("nan"), device=dev) for _ in range(2)]
    torch.cuda.synchronize()
    del poison                                     # the caching allocator hands these blocks to the next two allocations of n floats
    torch.cuda._sleep(400_000_000)                 # main stream busy for ~0.2 s: the zero fills below queue up behind it
    opt = nl.engine.FusedAdam([dict(param=torch.ones(16, device=dev), grad=torch.zeros(16, device=dev), lr=0.01),
                               dict(param=p, grad=g, lr=0.01, side=True)])
    opt.step(side_stream=side)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(p).all())
    torch.testing.assert_close(p, torch.full_like(p, 0.99), rtol=0, atol=1e-6)       # first Adam step: p - lr * sign(g)


def test_adam_ctl_reads_step_and_skip_from_the_device(nl):
    """nl_adam_*_ctl: the step count comes from the control block; a skipped iteration leaves parameter AND moments untouched
    (the reference `continue`s before optim.step(), render_helpers.py:405-409)."""
    dev = "cuda"
    cap, lib = nl._capi, nl._capi.lib()
    torch.manual_seed(3)
    n = 1000
    for dtype in (torch.float32, torch.bfloat16):
        p0 = (torch.randn(n, device=dev) * 0.05).to(dtype)
        g = torch.randn(n, device=dev)
        ctl = torch.zeros(cap.CTL_WORDS, dtype=torch.int32, device=dev)
        a = nl.engine.FusedAdam([dict(param=p0.clone(), grad=g, lr=0.01)])
        b = nl.engine.FusedAdam([dict(param=p0.clone(), grad=g, lr=0.01)], ctl=ctl)
        for step in (1, 2, 3):
            a.step()
            ctl[cap.CTL_ADAM_STEP] = step
            b.step()
            if step == 2:                      # an iteration without hits in between: nothing may move, the step count stays
                ctl[cap.CTL_SKIP_NOW] = 1
                before = [b.groups[0][k].clone() for k in ("param", "m", "v")]
                b.step()
                assert all(torch.equal(x, b.groups[0][k]) for x, k in zip(before, ("param", "m", "v")))
                ctl[cap.CTL_SKIP_NOW] = 0
        assert torch.equal(a.groups[0]["param"], b.groups[0]["param"])
        assert torch.equal(a.groups[0]["m"], b.groups[0]["m"]) and torch.equal(a.groups[0]["v"], b.groups[0]["v"])


def test_iter_status_folds_statistics(nl):
    cap, lib = nl._capi, nl._capi.lib()
    dev = "cuda"
    ctl = torch.zeros((2, cap.CTL_WORDS), dtype=torch.int32, device=dev)
    ctl[0, cap.CTL_MIN_HIT] = 2 ** 31 - 1
    seq = [dict(n_hit_rays=50, n_samples=700, error=0), dict(n_hit_rays=0, n_samples=0, error=0), dict(n_hit_rays=40, n_samples=900, error=2),
           dict(n_hit_rays=45, n_samples=100, error=1)]
    cur = 0
    for s in seq:
        st = cap.RenderStats()
        for k, v in s.items():
            setattr(st, k, v)
        d = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(dev)
        cap.check(lib.nl_iter_status(cap.ptr(d), cap.ptr(ctl[cur]), cap.ptr(ctl[cur ^ 1]), cap.stream_ptr()))
        cur ^= 1
    c = ctl[cur].tolist()
    assert c[cap.CTL_ERROR] == 3 and c[cap.CTL_SKIPPED] == 2 and c[cap.CTL_SKIP_NOW] == 1 and c[cap.CTL_ADAM_STEP] == 2
    assert c[cap.CTL_MIN_HIT] == 0 and c[cap.CTL_ITERS] == 4 and c[cap.CTL_MAX_SAMPLES] == 900


def test_stats_pack_kernels_match_the_host_layout(nl):
    """The CUDA pack/unpack kernels of the multi-GPU statistics exchange and the torch restatement used on CPU tensors (gloo tests)
    produce the same vector and the same unpacked struct."""
    cap = nl._capi
    nld = nl.dist
    world, rank = 4, 2
    st = cap.RenderStats()
    st.n_hit_rays, st.max_samples, st.error = 12345, 37, 2
    st.cnt_fs_valid, st.cnt_sdf_valid, st.pad_fs_rays, st.pad_fs_nsamp, st.pad_sdf_rays, st.pad_sdf_nsamp = 10 ** 10, 987654321, 77, 1234, 55, 999
    st.pad_sdf_d2, st.pad_sdf_d2_nsamp, st.fs_sum, st.sdf_sum = 1234.5678, 98765.4321, 3.14159265358979, 2.718281828459045e-3
    host = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).clone()
    devs = host.cuda()
    b_h = torch.empty(nld.stats_words(world), dtype=torch.float64)
    b_d = torch.empty(nld.stats_words(world), dtype=torch.float64, device="cuda")
    nld.pack_stats(host, b_h, rank, world, 0)
    nld.pack_stats(devs, b_d, rank, world, 0)
    assert torch.equal(b_h, b_d.cpu())
    # pretend the other ranks contributed: a larger S_max in slot 0, error bit 0 in slot 3
    for b in (b_h, b_d):
        b[:9] *= 3
        b[nld.FIXED + 0] = 41.0
        b[nld.FIXED + world + 3] = 1.0
    nld.unpack_stats(host, b_h, world, 0)
    nld.unpack_stats(devs, b_d, world, 0, 1.0, 10000.0)
    a, b = cap.RenderStats.from_buffer_copy(host.numpy().tobytes()), cap.RenderStats.from_buffer_copy(devs.cpu().numpy().tobytes())
    for k in ("n_hit_rays", "max_samples", "error", "cnt_fs_valid", "cnt_sdf_valid", "pad_fs_rays", "pad_fs_nsamp", "pad_sdf_rays", "pad_sdf_nsamp",
              "pad_sdf_d2", "pad_sdf_d2_nsamp"):
        assert getattr(a, k) == getattr(b, k), k
    assert b.max_samples == 41 and b.error == 3 and b.n_hit_rays == 3 * 12345
    assert b.g_fs > 0 and b.w_fs > 0                                    # the CUDA unpack re-derived the loss constants
    h_h, h_d = torch.zeros(4), torch.zeros(4, device="cuda")
    host2, dev2 = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).clone(), torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).cuda()
    nld.pack_stats(host2, h_h, 0, world, 1)
    nld.pack_stats(dev2, h_d, 0, world, 1)
    assert torch.equal(h_h, h_d.cpu())
    nld.unpack_stats(dev2, h_d, world, 1)
    c = cap.RenderStats.from_buffer_copy(dev2.cpu().numpy().tobytes())
    assert abs(c.fs_sum - st.fs_sum) < 1e-13 * st.fs_sum + 1e-15 and abs(c.sdf_sum - st.sdf_sum) < 1e-13


def test_select_rays_is_a_uniform_subset_in_point_order(nl):
    """nl_select_rays (LidarFrame.sample_rays on the device): exactly N distinct points per scan, ascending, gathered correctly, every
    point equally likely (chi-square over many draws), also when more than half of the points are wanted (complement path) and for
    several scans of different length in one launch."""
    rh = nl.render_helpers
    dev = torch.device("cuda")
    torch.manual_seed(0)
    F, cap = 3, 5000
    n = torch.tensor([5000, 3777, 64], dtype=torch.int64, device=dev)
    dirs = torch.randn(F, cap, 3, device=dev)
    gt = torch.arange(F * cap, device=dev, dtype=torch.float32).view(F, cap)             # gt[f, i] identifies the point
    cos = -gt
    for N in (64, 1000):
        counts = torch.zeros(F, cap, device=dev)
        draws = 300
        for it in range(draws):
            seed = torch.tensor([it * 7919 + 1], dtype=torch.int32, device=dev)
            d, g, c = rh.select_rays_device(dirs, gt, cos, N, n_dev=n, seed=seed)
            g = g.view(F, N)
            for f in range(F):
                k = min(N, int(n[f]))
                idx = (g[f, :k] - f * cap).long()
                assert bool((idx[1:] > idx[:-1]).all()) and int(idx.min()) >= 0 and int(idx.max()) < int(n[f])      # distinct, ascending, in range
                assert torch.equal(d.view(F, N, 3)[f, :k], dirs[f, idx]) and torch.equal(c.view(F, N)[f, :k], cos[f, idx])
                counts[f, idx] += 1
        for f in range(2):                                   # (the third scan has exactly 64 points: always all of them)
            nf = int(n[f])
            p = N / nf
            x = counts[f, :nf]
            z = (x - draws * p) / (draws * p * (1 - p)) ** 0.5
            assert abs(float(z.mean())) < 0.05 and 0.9 < float(z.std()) < 1.1, (N, f, float(z.mean()), float(z.std()))
        assert bool((counts[2, :64] == draws).all())
    # different seeds give different subsets, the same seed the same subset
    s1 = torch.tensor([5], dtype=torch.int32, device=dev)
    a = rh.select_rays_device(dirs, gt, cos, 100, n_dev=n, seed=s1)[1].clone()
    b = rh.select_rays_device(dirs, gt, cos, 100, n_dev=n, seed=s1)[1].clone()
    c2 = rh.select_rays_device(dirs, gt, cos, 100, n_dev=n, seed=torch.tensor([6], dtype=torch.int32, device=dev))[1]
    assert torch.equal(a[:264], b[:264]) and not torch.equal(a[:100], c2[:100])     # (scan 3 has only 64 points: its last 36 slots stay unwritten)


def _select_keys_torch(seed, f, n, dev):
    """The key generator of csrc/select.cu restated with int64 torch ops: key(i) = mix32(seed_f ^ mix32(i * 0x9E3779B1 + 0x7F4A7C15))."""
    M = 0xFFFFFFFF

    def mix(x):
        x = x ^ (x >> 16); x = (x * 0x7FEB352D) & M; x = x ^ (x >> 15); x = (x * 0x846CA68B) & M; return x ^ (x >> 16)

    sf = mix(torch.tensor([(seed ^ ((0x9E3779B9 * (f + 1)) & M)) & M], dtype=torch.int64, device=dev))
    i = torch.arange(n, dtype=torch.int64, device=dev)
    return mix(sf ^ mix((i * 0x9E3779B1 + 0x7F4A7C15) & M))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2048, 70000])
def test_select_rays_equals_top_n_of_the_hashed_keys_at_scan_size(nl, N):
    """At the size of a real scan (10^5 points, several scans per launch) the kernel's subset is exactly the N smallest keys
    (ties to the lower index) -- the radix select, the cluster-wide histograms and the ordered emission against torch's sort."""
    rh = nl.render_helpers
    dev = torch.device("cuda")
    F, cap = 5, 262144          # scans above 131 072 points take the kernel's re-hashing path, smaller ones keep their keys in registers
    n = torch.tensor([262144, 200003, 131072, 65537, 1500], dtype=torch.int64, device=dev)
    dirs = torch.randn(F, cap, 3, device=dev)
    gt = torch.arange(F * cap, device=dev, dtype=torch.float32).view(F, cap)
    for seed in (1, 0x7FFFFFF1, 424242):
        idx = torch.full((F * N,), -1, dtype=torch.int32, device=dev)
        out = (torch.empty(F * N, 3, device=dev), torch.empty(F * N, device=dev), torch.empty(F * N, device=dev))
        sd = torch.tensor([seed], dtype=torch.int32, device=dev)
        nl._capi.check(nl._capi.lib().nl_select_rays(F, cap, N, nl._capi.ptr(n), nl._capi.ptr(sd), 0, nl._capi.ptr(dirs), nl._capi.ptr(gt), nl._capi.ptr(gt),
                                                     nl._capi.ptr(out[0]), nl._capi.ptr(out[1]), nl._capi.ptr(out[2]), nl._capi.ptr(idx), nl._capi.stream_ptr()),
                       "nl_select_rays")
        for f in range(F):
            nf = int(n[f]); k = min(N, nf)
            key = _select_keys_torch(seed, f, nf, dev)
            want = torch.sort(torch.topk((key << 24) | torch.arange(nf, device=dev), k, largest=False).indices).values
            got = idx.view(F, N)[f, :k].long()
            assert torch.equal(got, want), (seed, f, int((got != want).sum()))
            assert torch.equal(out[1].view(F, N)[f, :k], gt[f, want]) and torch.equal(out[0].view(F, N, 3)[f, :k], dirs[f, want])

