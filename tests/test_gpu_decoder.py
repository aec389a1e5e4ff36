"""The SDF decoder kernels (csrc/mlp_tc.cu: tcgen05 3xTF32, width 256; csrc/mlp.cu: fp32 CUDA cores, widths 32..256) against an
fp64 evaluation of the same function, element by element.

Yardstick: the same fp64 computation run again on absolute values (|W|, |b|, |x|, |d sdf|, forward magnitudes) gives, for every
output element, the sum of the absolute values of its terms, A.  A kernel passes when |kernel - fp64| <= 2^-16 A everywhere.
2^-16 is far above what fp32 or 3xTF32 rounding can produce and about 30x below the error of single-pass TF32, so a dropped lo
term, a wrong or stale row, a missed tile or a wrong loss coefficient all fail.  Input rows with a pre-activation within 2^-13 A
of a ReLU kink are dropped when drawn, so the kernel and the reference agree on every relu' and every row compares directly.

Shapes sit at the tile edges of the persistent kernels (128-sample tiles, one CTA per SM of a 148-SM B200) and at the size of a
full scan (~700 k samples: ~37 tiles per CTA, the weight-gradient rings wrap hundreds of times).  Run with -s to see, per
scenario, the largest err / A and how many drawn rows were dropped near kinks.
"""
import ctypes as C
import math

import pytest
import torch

from util import golden, load_decoder

pytestmark = pytest.mark.gpu

N_SM = 148                  # B200: the persistent decoder kernels run one CTA per SM
TILE = 128                  # samples per tile in both implementations
FULL_SCAN = 700_000         # samples of one full LiDAR scan
TOL = 2.0 ** -16            # pass bound, relative to A
NOTE = 2.0 ** -18           # ratios above this are flagged in the printed table
KINK = 2.0 ** -13           # drop rows with |pre-activation| < KINK * A (8x above TOL)
SENT = -7.4e33              # sentinel for rows past the device-side sample count
GRAD_NAMES = ("gW0", "gb0", "gW1", "gb1", "gW2", "gb2")   # order of DecoderBuffers.params / .grads
CHUNK = 1 << 17             # rows per fp64 chunk (bounds the reference's memory at full-scan size)

GOLDEN_DECODERS = {"render": ("render.npz", "dec_", 256), "map_dec0": ("mapping_tracking.npz", "map_dec0_", 256),
                   "map_dec_after": ("mapping_tracking.npz", "map_dec_after_", 256), "w32": ("chain.npz", "w32_p_", 32)}
DECODERS = {256: ("render", "map_dec0", "map_dec_after"), 128: ("seed128",), 64: ("seed64",), 32: ("w32",)}


@pytest.fixture(scope="module")
def nl():
    import nerfloam_b200 as nl
    assert torch.cuda.is_available()
    return nl


_dec_cache = {}


def decoder(nl, name):
    """Golden decoders, or nn.Linear's default initialisation under a fixed seed ("seed<width>")."""
    if name not in _dec_cache:
        if name.startswith("seed"):
            W = int(name[4:])
            torch.manual_seed(W)
            dec = nl.lidar.Decoder(depth=2, width=W, in_dim=16, skips=[], embedder="none", multires=0).cuda()
        else:
            f, prefix, W = GOLDEN_DECODERS[name]
            dec = load_decoder(golden(f), prefix, width=W)
        _dec_cache[name] = dec
    return _dec_cache[name]


def buffers(nl, name):
    bufs = nl.engine.DecoderBuffers(decoder(nl, name), torch.device("cuda"))
    bufs.refresh_transposes()
    return bufs


# ------------------------------------------------------------------------------------------------ fp64 reference
def _fused_dsdf(sdf, A_sdf, loss, rows):
    """d loss / d sdf of the fused loss (criterion.py, mlp.cu / mlp_tc.cu) in fp64, with its yardstick: the terms of the
    expression plus what the error of sdf carries into it."""
    fl = loss["flag"][rows].long()
    f1, f2 = (fl & 1).bool().double(), (fl & 2).bool().double()
    r = loss["ray"][rows].long()
    cos = loss["cos"][r] if loss["cos"] is not None else torch.ones_like(loss["depth"][rows])
    z = (loss["depth"][rows] * cos).double()          # the kernel forms z in fp32
    gt = loss["gt"][r].double()
    t, g_fs, g_sdf = loss["t"], loss["g_fs"], loss["g_sdf"]
    e1, A_e1 = sdf - 1.0, sdf.abs() + 1.0 + A_sdf
    e2, A_e2 = z + t * sdf - gt, z.abs() + t * sdf.abs() + gt.abs() + t * A_sdf
    d = 2 * g_fs * e1 * f1 + 2 * g_sdf * t * e2 * f2
    A_d = 2 * abs(g_fs) * A_e1 * f1 + 2 * abs(g_sdf) * t * A_e2 * f2
    sums = {"fs_sum": ((e1 * e1 * f1).sum(), ((e1 * e1 + 2 * e1.abs() * A_e1) * f1).sum()),
            "sdf_sum": ((e2 * e2 * f2).sum(), ((e2 * e2 + 2 * e2.abs() * A_e2) * f2).sum())}
    return d, A_d, sums


def ref64(x, params, dsdf=None, loss=None):
    """fp64 decoder on rows x [M,16]: {output: (value, A)} for sdf and -- with dsdf [M] or the fused loss inputs -- d x, the six
    parameter gradients and the loss sums; "kink": rows with a pre-activation within KINK * A of 0."""
    W0, b0, W1, b1, w2, b2 = [p.detach().double() for p in params]
    w2, b2 = w2.reshape(-1), b2.reshape(())
    aW0, ab0, aW1, ab1, aw2, ab2 = W0.abs(), b0.abs(), W1.abs(), b1.abs(), w2.abs(), b2.abs()
    train = dsdf is not None or loss is not None
    rows_out = {k: ([], []) for k in (("sdf", "dx") if train else ("sdf",))}
    kinks = []
    acc = {}

    def add(k, v, a):
        if k in acc:
            acc[k][0].add_(v)
            acc[k][1].add_(a)
        else:
            acc[k] = (v.clone(), a.clone())

    for s in range(0, x.shape[0], CHUNK):
        rows = slice(s, s + CHUNK)
        xs = x[rows].double()
        ax = xs.abs()
        a1, A1 = xs @ W0.T + b0, ax @ aW0.T + ab0
        m1 = a1 > 0
        k1 = (a1.abs() < KINK * A1).any(1)
        h1, H1 = a1 * m1, A1 * m1
        del a1, A1
        a2, A2 = h1 @ W1.T + b1, H1 @ aW1.T + ab1
        m2 = a2 > 0
        kinks.append(k1 | (a2.abs() < KINK * A2).any(1))
        h2, H2 = a2 * m2, A2 * m2
        del a2, A2
        sdf, A_sdf = h2 @ w2 + b2, H2 @ aw2 + ab2
        rows_out["sdf"][0].append(sdf)
        rows_out["sdf"][1].append(A_sdf)
        if not train:
            continue
        if dsdf is not None:
            d = dsdf[rows].double()
            A_d = d.abs()
        else:
            d, A_d, sums = _fused_dsdf(sdf, A_sdf, loss, rows)
            for k, (v, a) in sums.items():
                add(k, v, a)
        dh2, A_dh2 = d[:, None] * (w2 * m2), A_d[:, None] * (aw2 * m2)
        dh1, A_dh1 = (dh2 @ W1) * m1, (A_dh2 @ aW1) * m1
        rows_out["dx"][0].append(dh1 @ W0)
        rows_out["dx"][1].append(A_dh1 @ aW0)
        add("gW0", dh1.T @ xs, A_dh1.T @ ax)
        add("gb0", dh1.sum(0), A_dh1.sum(0))
        add("gW1", dh2.T @ h1, A_dh2.T @ H1)
        add("gb1", dh2.sum(0), A_dh2.sum(0))
        add("gW2", d @ h2, A_d @ H2)
        add("gb2", d.sum(), A_d.sum())
    out = {k: (torch.cat(v), torch.cat(a)) for k, (v, a) in rows_out.items()}
    out.update(acc)
    out["kink"] = torch.cat(kinks)
    if train and "fs_sum" not in out:          # external d sdf: the kernel leaves the loss sums alone
        z = torch.zeros((), dtype=torch.float64, device=x.device)
        out["fs_sum"] = out["sdf_sum"] = (z, z)
    return out


def draw_rows(params, M, regime, gen):
    """M input rows: x ~ N(0, 0.05^2) ("small", the gather's range) or N(0, 1) ("unit"), with a block of all-zero rows across the
    middle; rows near a ReLU kink are dropped and redrawn.  Returns x and a note on how many rows were dropped."""
    scale = {"small": 0.05, "unit": 1.0}[regime]
    dev = torch.device("cuda")
    nz = min(64, M // 4)
    zero = torch.zeros((nz, 16), device=dev)
    zero_note = ""
    if nz and bool(ref64(zero[:1], params)["kink"][0]):
        nz, zero = 0, zero[:0]
        zero_note = ", zero rows sit on a kink: block left out"
    need, parts, have, drawn = M - nz, [], 0, 0
    while have < need:
        n = max(2 * (need - have), 256)
        c = torch.randn((n, 16), generator=gen, device=dev) * scale
        c = c[~ref64(c, params)["kink"]]
        drawn += n
        parts.append(c)
        have += c.shape[0]
    x = torch.cat(parts)[:need] if parts else torch.zeros((0, 16), device=dev)
    kept = sum(p.shape[0] for p in parts)
    pos = need // 2
    x = torch.cat([x[:pos], zero, x[pos:]]).contiguous()
    return x, f"dropped {drawn - kept}/{drawn} {regime} rows{zero_note}"


def loss_inputs(M, gen, with_cos):
    """Per-sample inputs of the fused loss: s_flag in {0,1,2,3} mixed, random rays, depths near the ray's measured depth."""
    dev = torch.device("cuda")
    R = M // 8 + 1
    ray = torch.randint(0, R, (M,), generator=gen, device=dev, dtype=torch.int32)
    flag = torch.randint(0, 4, (M,), generator=gen, device=dev, dtype=torch.int32).to(torch.uint8)
    cos = (0.5 + 0.5 * torch.rand(R, generator=gen, device=dev)) if with_cos else None
    gt = 2.0 + 18.0 * torch.rand(R, generator=gen, device=dev)
    z = gt[ray.long()] + 0.3 * torch.randn(M, generator=gen, device=dev)
    depth = (z / cos[ray.long()] if with_cos else z).contiguous()
    f32 = lambda v: float(torch.tensor(v, dtype=torch.float32))   # noqa: E731  the kernel sees these as fp32
    return dict(flag=flag, depth=depth, ray=ray, cos=cos, gt=gt, t=f32(0.3), g_fs=f32(0.5), g_sdf=f32(40.0))


def stats_block(nl, loss, fs_sum=0.0, sdf_sum=0.0):
    st = nl._capi.RenderStats()
    st.g_fs, st.g_sdf, st.fs_sum, st.sdf_sum = loss["g_fs"], loss["g_sdf"], fs_sum, sdf_sum
    return torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).cuda()


def read_stats(nl, t):
    return nl._capi.RenderStats.from_buffer_copy(t.cpu().numpy().tobytes())


def run_train(nl, bufs, M_cap, x, sdf, dx, act, M_dev=None, dsdf=None, loss=None, stats=None, wgrad_stream=None):
    kw = dict(dsdf_ext=dsdf, wgrad_stream=wgrad_stream)
    if loss is not None:
        kw.update(s_flag=loss["flag"], s_depth=loss["depth"], s_ray=loss["ray"], cos=loss["cos"], gt_depth=loss["gt"],
                  stats_ptr=C.c_void_p(stats.data_ptr()), truncation=loss["t"])
    nl.engine.mlp_train(bufs, M_cap, M_dev, x, sdf, dx, act is not None, act, **kw)


# ------------------------------------------------------------------------------------------------ comparison
class Yardstick:
    """Collects |kernel - fp64| / A per output; prints the worst ratio of the scenario and fails on any element over TOL."""

    def __init__(self, label):
        self.label, self.worst, self.fail, self.notes = label, {}, [], []

    def cmp(self, name, got, ref, A, base=None):
        """got ~ base + ref (base: what the output held before the kernel accumulated into it)."""
        got = got.detach().double().reshape(ref.shape)
        A = A.double()
        if base is not None:
            ref = ref + base.double().reshape(ref.shape)
            A = A + base.double().reshape(ref.shape).abs()
        err = (got - ref).abs()
        ok = err <= TOL * A                      # NaN fails
        ratio = torch.where(A > 0, err / A.clamp_min(1e-300), torch.where(err == 0, 0.0, math.inf)).nan_to_num(nan=math.inf)
        w = float(ratio.max()) if ratio.numel() else 0.0
        self.worst[name] = max(self.worst.get(name, 0.0), w)
        if not bool(ok.all()):
            bad = (~ok).reshape(-1)
            i = int(bad.nonzero()[0])
            self.fail.append(f"{name}: {int(bad.sum())}/{bad.numel()} elements over 2^-16 A, worst err/A {w:.3g}; first at flat index {i}: "
                             f"kernel {float(got.reshape(-1)[i]):.9g}, fp64 {float(ref.reshape(-1)[i]):.9g}, A {float(A.reshape(-1)[i]):.3g}")

    def cmp_all(self, ref, sdf=None, dx=None, grads=None, stats=None, grad_base=None, stats_base=(0.0, 0.0)):
        if sdf is not None:
            self.cmp("sdf", sdf, *ref["sdf"])
        if dx is not None:
            self.cmp("dx", dx, *ref["dx"])
        if grads is not None:
            for k, (name, g) in enumerate(zip(GRAD_NAMES, grads)):
                self.cmp(name, g, *ref[name], base=None if grad_base is None else grad_base[k])
        if stats is not None:
            dev = ref["sdf"][0].device
            for name, base in zip(("fs_sum", "sdf_sum"), stats_base):
                self.cmp(name, torch.tensor(getattr(stats, name), dtype=torch.float64, device=dev), *ref[name],
                         base=torch.tensor(base, dtype=torch.float64, device=dev))

    def exact(self, what, cond):
        if not cond:
            self.fail.append(what)

    def finish(self):
        name, w = max(self.worst.items(), key=lambda kv: kv[1]) if self.worst else ("-", 0.0)
        flag = "   <-- above 2^-18" if w > NOTE else ""
        print(f"\n[decoder vs fp64] {self.label}: max err/A {w:.2e} ({name}){flag}" + "".join(f"; {n}" for n in self.notes))
        assert not self.fail, self.label + ":\n  " + "\n  ".join(self.fail)


def free_cuda():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ tests
EDGE_M = (1, 127, 128, 129, N_SM * TILE - 1, N_SM * TILE, N_SM * TILE + 1, 3 * N_SM * TILE + 37)
FWD_CASES = [("tc", 256, M) for M in EDGE_M + (FULL_SCAN,)] + [("simt", W, M) for W in (32, 64, 128, 256) for M in EDGE_M]


@pytest.mark.parametrize("impl,width,M", FWD_CASES)
def test_forward_vs_fp64(nl, monkeypatch, impl, width, M):
    """sdf of nl_mlp_tc_forward / nl_mlp_forward, element by element, for every decoder of the width and both input regimes."""
    monkeypatch.setenv("NL_MLP_IMPL", impl)
    ys = Yardstick(f"forward {impl}@{width} M={M}")
    gen = torch.Generator(device="cuda").manual_seed(1000 + M)
    for name in DECODERS[width]:
        bufs = buffers(nl, name)
        for regime in ("small", "unit"):
            x, note = draw_rows(bufs.params, M, regime, gen)
            ys.notes.append(f"{name}: {note}")
            sdf = torch.full((M,), math.nan, device="cuda")
            nl.engine.mlp_forward(bufs, M, None, x, sdf)
            ys.cmp_all(ref64(x, bufs.params), sdf=sdf)
            del x, sdf
    if M == FULL_SCAN:
        free_cuda()
    ys.finish()


TRAIN_IMPLS = (("tc", 256), ("simt", 32), ("simt", 64), ("simt", 128), ("simt", 256))
LOSSES = ("ext", "fused_cos", "fused_nocos")
TRAIN_CASES = [(impl, W, wgrad, loss, M) for impl, W in TRAIN_IMPLS for wgrad in (False, True) for loss in LOSSES
               for M in (129, N_SM * TILE + 77)] + [("tc", 256, True, loss, FULL_SCAN) for loss in ("ext", "fused_cos")]


def make_loss(nl, mode, M, gen, fs_sum=0.0, sdf_sum=0.0):
    """(dsdf_ext, loss inputs, stats block) for a loss mode."""
    if mode == "ext":
        return (0.1 * torch.randn(M, generator=gen, device="cuda")).contiguous(), None, None
    loss = loss_inputs(M, gen, with_cos=(mode == "fused_cos"))
    return None, loss, stats_block(nl, loss, fs_sum, sdf_sum)


@pytest.mark.parametrize("impl,width,wgrad,loss_mode,M", TRAIN_CASES)
def test_train_vs_fp64(nl, monkeypatch, impl, width, wgrad, loss_mode, M):
    """nl_mlp_tc_train / nl_mlp_train: sdf, d x, the six decoder gradients and the loss sums against fp64."""
    monkeypatch.setenv("NL_MLP_IMPL", impl)
    ys = Yardstick(f"train {impl}@{width} wgrad={wgrad} {loss_mode} M={M}")
    gen = torch.Generator(device="cuda").manual_seed(2000 + M)
    regimes = ("small",) if M == FULL_SCAN else ("small", "unit")
    for name in DECODERS[width]:
        bufs = buffers(nl, name)
        for regime in regimes:
            x, note = draw_rows(bufs.params, M, regime, gen)
            ys.notes.append(f"{name}: {note}")
            dsdf, loss, stats = make_loss(nl, loss_mode, M, gen)
            sdf = torch.full((M,), math.nan, device="cuda")
            dx = torch.full((M, 16), math.nan, device="cuda")
            act = nl.engine.alloc_act(width, M, "cuda") if wgrad else None
            bufs.gradflat.zero_()
            run_train(nl, bufs, M, x, sdf, dx, act, dsdf=dsdf, loss=loss, stats=stats)
            ref = ref64(x, bufs.params, dsdf=dsdf, loss=loss)
            ys.cmp_all(ref, sdf=sdf, dx=dx, grads=bufs.grads if wgrad else None, stats=read_stats(nl, stats) if stats is not None else None)
            if not wgrad:
                ys.exact("gradient buffers written without wgrad", bool((bufs.gradflat == 0).all()))
            del x, sdf, dx, act, ref, dsdf, loss
            if M == FULL_SCAN:
                free_cuda()
    ys.finish()


M_CAP = 3 * N_SM * TILE + 37
DEV_COUNTS = (0, 1, 128, 129, M_CAP - 1, M_CAP, M_CAP + 1000)


@pytest.mark.parametrize("loss_mode", ("ext", "fused_cos"))
@pytest.mark.parametrize("wgrad", (False, True))
@pytest.mark.parametrize("impl,width", (("tc", 256), ("simt", 256), ("simt", 64)))
def test_device_side_sample_count(nl, monkeypatch, impl, width, wgrad, loss_mode):
    """Capacity on the host, count on the device (as SDFEngine calls the decoder): rows past the device count are neither read
    (they hold NaN: features, d sdf, depths and the whole weight-gradient scratch) nor written (sdf / d x keep a sentinel bit
    for bit); a count above the capacity is clamped to it; a count of 0 leaves gradients and loss sums bit for bit unchanged."""
    monkeypatch.setenv("NL_MLP_IMPL", impl)
    ys = Yardstick(f"device count {impl}@{width} wgrad={wgrad} {loss_mode} M_cap={M_CAP}")
    gen = torch.Generator(device="cuda").manual_seed(3000 + width)
    name = DECODERS[width][0]
    bufs = buffers(nl, name)
    x_all, note = draw_rows(bufs.params, M_CAP, "small", gen)
    ys.notes.append(note)
    dsdf_all, loss_all, _ = make_loss(nl, loss_mode, M_CAP, gen)
    sent_bits = torch.tensor(SENT, dtype=torch.float32).view(torch.int32)
    m_dev = torch.zeros(1, dtype=torch.int32, device="cuda")
    for count in DEV_COUNTS:
        n = min(count, M_CAP)
        feats = x_all.clone()
        feats[n:] = math.nan
        dsdf = loss = None
        if dsdf_all is not None:
            dsdf = dsdf_all.clone()
            dsdf[n:] = math.nan
        else:
            loss = dict(loss_all, flag=loss_all["flag"].clone(), depth=loss_all["depth"].clone())
            loss["flag"][n:] = 3
            loss["depth"][n:] = math.nan
        stats_base = (1.25, 3.5)
        stats = stats_block(nl, loss, *stats_base) if loss is not None else None
        sdf = torch.full((M_CAP,), SENT, device="cuda")
        dx = torch.full((M_CAP, 16), SENT, device="cuda")
        act = None
        if wgrad:
            act = nl.engine.alloc_act(width, M_CAP, "cuda")
            for t in act.values():
                t.fill_(math.nan)
        torch.manual_seed(count)
        grad_base = [torch.randn_like(g) * 0.01 for g in bufs.grads]
        for g, b in zip(bufs.grads, grad_base):
            g.copy_(b)
        m_dev.fill_(count)
        run_train(nl, bufs, M_CAP, feats, sdf, dx, act, M_dev=nl._capi.ptr(m_dev), dsdf=dsdf, loss=loss, stats=stats)
        sdf_f = torch.full((M_CAP,), SENT, device="cuda")
        nl.engine.mlp_forward(bufs, M_CAP, nl._capi.ptr(m_dev), feats, sdf_f)
        torch.cuda.synchronize()
        tag = f"M_dev={count}"
        ys.exact(f"{tag}: sdf rows >= {n} overwritten", bool((sdf[n:].view(torch.int32) == sent_bits).all()))
        ys.exact(f"{tag}: d x rows >= {n} overwritten", bool((dx[n:].view(torch.int32) == sent_bits).all()))
        ys.exact(f"{tag}: forward sdf rows >= {n} overwritten", bool((sdf_f[n:].view(torch.int32) == sent_bits).all()))
        st = read_stats(nl, stats) if stats is not None else None
        if n == 0:
            if wgrad:
                for nm, g, b in zip(GRAD_NAMES, bufs.grads, grad_base):
                    ys.exact(f"{tag}: {nm} changed", torch.equal(g.view(torch.int32), b.view(torch.int32)))
            if st is not None:
                ys.exact(f"{tag}: loss sums changed ({st.fs_sum}, {st.sdf_sum})", (st.fs_sum, st.sdf_sum) == stats_base)
        else:
            sub_loss = None
            if loss is not None:
                sub_loss = dict(loss, flag=loss["flag"][:n], depth=loss["depth"][:n], ray=loss["ray"][:n])
            ref = ref64(x_all[:n], bufs.params, dsdf=None if dsdf is None else dsdf[:n], loss=sub_loss)
            ys.cmp_all(ref, sdf=sdf[:n], dx=dx[:n], grads=bufs.grads if wgrad else None, stats=st, grad_base=grad_base, stats_base=stats_base)
            ys.cmp("forward sdf", sdf_f[:n], *ref["sdf"])
        if not wgrad:
            for nm, g, b in zip(GRAD_NAMES, bufs.grads, grad_base):
                ys.exact(f"{tag}: {nm} written without wgrad", torch.equal(g, b))
        del feats, dsdf, loss, stats, sdf, dx, act, sdf_f
    ys.finish()


def test_single_sample_impulse_full_scan(nl, monkeypatch):
    """tc with weight gradients at full-scan size, d sdf one-hot at tile / grid edges: every gradient is that one sample's fp64
    outer products (A = that sample's own terms), so a dropped, duplicated or stale row shows even though M is 700 k.  An
    all-zero d sdf gives gradients and d x of exactly 0."""
    monkeypatch.setenv("NL_MLP_IMPL", "tc")
    M = FULL_SCAN
    ys = Yardstick(f"impulse tc@256 M={M}")
    gen = torch.Generator(device="cuda").manual_seed(4000)
    bufs = buffers(nl, "map_dec_after")
    x, note = draw_rows(bufs.params, M, "small", gen)
    ys.notes.append(note)
    act = nl.engine.alloc_act(256, M, "cuda")
    sdf = torch.empty(M, device="cuda")
    dx = torch.empty((M, 16), device="cuda")
    dsdf = torch.zeros(M, device="cuda")
    for p in (None, 0, 127, 128, N_SM * TILE - 1, N_SM * TILE, M - 1):
        dsdf.zero_()
        if p is not None:
            dsdf[p] = 0.75
        sdf.fill_(math.nan)
        dx.fill_(math.nan)
        bufs.gradflat.zero_()
        run_train(nl, bufs, M, x, sdf, dx, act, dsdf=dsdf)
        torch.cuda.synchronize()
        if p is None:
            ys.cmp_all(ref64(x, bufs.params), sdf=sdf)
            ys.exact("zero d sdf: d x not exactly 0", bool((dx == 0).all()))
            for nm, g in zip(GRAD_NAMES, bufs.grads):
                ys.exact(f"zero d sdf: {nm} not exactly 0", bool((g == 0).all()))
            free_cuda()
            continue
        ref = ref64(x[p:p + 1], bufs.params, dsdf=dsdf[p:p + 1])
        ys.cmp_all(ref, dx=dx[p:p + 1], grads=bufs.grads)
        others = torch.ones(M, dtype=torch.bool, device="cuda")
        others[p] = False
        ys.exact(f"impulse at {p}: d x of other rows not exactly 0", bool((dx[others] == 0).all()))
    del x, act, sdf, dx, dsdf
    free_cuda()
    ys.finish()


@pytest.mark.parametrize("impl,width", (("tc", 256), ("simt", 256), ("simt", 64)))
def test_gradients_and_loss_accumulate(nl, monkeypatch, impl, width):
    """Gradients accumulate into bufs.grads and the loss into stats: non-zero buffers end as prefill + fp64."""
    monkeypatch.setenv("NL_MLP_IMPL", impl)
    M = N_SM * TILE + 77
    ys = Yardstick(f"accumulate {impl}@{width} M={M}")
    gen = torch.Generator(device="cuda").manual_seed(5000 + width)
    bufs = buffers(nl, DECODERS[width][-1])
    x, note = draw_rows(bufs.params, M, "small", gen)
    ys.notes.append(note)
    stats_base = (17.0625, 0.4375)
    _, loss, stats = make_loss(nl, "fused_cos", M, gen, *stats_base)
    ref = ref64(x, bufs.params, loss=loss)
    # prefill at the gradients' own scale, so that overwriting or a double add shows as an O(1) error
    grad_base = [(torch.randn(g.shape, generator=gen, device="cuda") * ref[nm][0].abs().max()).float() for nm, g in zip(GRAD_NAMES, bufs.grads)]
    for g, b in zip(bufs.grads, grad_base):
        g.copy_(b)
    sdf = torch.empty(M, device="cuda")
    dx = torch.empty((M, 16), device="cuda")
    run_train(nl, bufs, M, x, sdf, dx, nl.engine.alloc_act(width, M, "cuda"), loss=loss, stats=stats)
    ys.cmp_all(ref, sdf=sdf, dx=dx, grads=bufs.grads, stats=read_stats(nl, stats), grad_base=grad_base, stats_base=stats_base)
    ys.finish()


def test_weight_gradient_side_stream(nl, monkeypatch):
    """tc weight-gradient kernels on a second stream (as SDFEngine.forward_backward runs them): ordered behind the gradient
    prefill on the main stream, joined the same way, and equal to the single-stream result and to fp64."""
    monkeypatch.setenv("NL_MLP_IMPL", "tc")
    M = 3 * N_SM * TILE + 37
    ys = Yardstick(f"weight-gradient stream tc@256 M={M}")
    gen = torch.Generator(device="cuda").manual_seed(6000)
    bufs = buffers(nl, "map_dec0")
    x, note = draw_rows(bufs.params, M, "small", gen)
    ys.notes.append(note)
    _, loss, _ = make_loss(nl, "fused_cos", M, gen)
    ref = ref64(x, bufs.params, loss=loss)
    side = torch.cuda.Stream()
    results = {}
    for mode in ("single", "side"):
        stats = stats_block(nl, loss)
        act = nl.engine.alloc_act(256, M, "cuda")
        sdf = torch.empty(M, device="cuda")
        dx = torch.empty((M, 16), device="cuda")
        bufs.gradflat.fill_(math.nan)
        bufs.gradflat.zero_()
        run_train(nl, bufs, M, x, sdf, dx, act, loss=loss, stats=stats, wgrad_stream=side if mode == "side" else None)
        if mode == "side":
            torch.cuda.current_stream().wait_stream(side)   # engine.forward_backward: gradients complete before they are used
        g = [t.clone() for t in bufs.grads]
        torch.cuda.synchronize()
        ys.cmp_all(ref, sdf=sdf, dx=dx, grads=g, stats=read_stats(nl, stats))
        results[mode] = g
    for nm, a, b, (_, A) in zip(GRAD_NAMES, results["side"], results["single"], (ref[n] for n in GRAD_NAMES)):
        ys.exact(f"{nm}: side-stream and single-stream results differ by more than 2^-16 A",
                 bool(((a.double() - b.double()).abs() <= TOL * A).all()))
    ys.finish()
