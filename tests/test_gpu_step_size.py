"""The persistent and grid-strided kernels at the training step's batch size (B = 512 segments per encoder call), against
plain fp64 references evaluated on the GPU.

The launch code sizes its grids to the problem, so at the small shapes of test_gpu_parity.py almost every CTA or thread
gets exactly one unit of work: one GEMM tile (K6), at most three rows (K5), one segment (the k-NN self kernel).  The code
that runs only from the second unit on - the second TMEM accumulator buffer and its barrier phases, the moments carried
across tiles, the 4-row unrolled loops, the L2-hint split, the TMA ring across segment boundaries - is what this module
reaches.  Each test first checks, with a Python mirror of the launch geometry, that its shape really gives every CTA or
thread several units; a larger GPU or a changed launch rule then fails loudly instead of shrinking the coverage back.

Element-wise bounds are derived in the docstrings.  The module prints, at teardown, the largest measured error of each
kernel family as a fraction of its bound, the peak device memory and the wall time.
"""
import math
import time

import pytest
import torch

import golden_io as gio
from golden_io import _default_kernel_options, _exact_fp32_library_math  # noqa: F401  (autouse: TF32 off, default options)
from grafp_b200 import ops, synth
from grafp_b200.encoder.graph_encoder import GraphEncoder
from oracle import grafp_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
B_STEP = 512                                      # segments per encoder call of the training step (bench.py)
STAGES = [(1024, 64), (512, 128), (256, 256), (128, 512)]
U32 = 2.0 ** -24                                  # unit roundoff of fp32
U_BF16 = 2.0 ** -8                                # unit roundoff of bf16 (8 significant bits)
U_TF32 = 2.0 ** -10                               # TF32 keeps 10 explicit mantissa bits (bound holds for truncation)
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}

_WORST = {}                                       # kernel family -> largest (error / bound) seen


def _note(family, ratio):
    _WORST[family] = max(_WORST.get(family, 0.0), float(ratio))


def _ratio(err, bound):
    """max(err / bound) where 0 / 0 counts as 0: an element whose bound is zero (e.g. the gradient of a channel the
    ReLU masks completely) must come out exact, and any error there is an infinite ratio."""
    return float(torch.where(err == 0, torch.zeros_like(err), err / bound).max())


@pytest.fixture(scope="module", autouse=True)
def _report_and_release():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    peak = torch.cuda.max_memory_allocated() / 2 ** 30
    worst = ", ".join(f"{k} {v:.3g}" for k, v in sorted(_WORST.items()))
    print(f"\n[step-size] {torch.cuda.get_device_name()}: {time.time() - t0:.0f} s, peak {peak:.1f} GiB allocated; "
          f"largest error / bound: {worst}")
    torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _rows(t):
    """(B, C, N, 1) node rows as a (B * N, C) view."""
    B, C, N, _ = t.shape
    return t.permute(0, 2, 3, 1).reshape(B * N, C)


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


# ------------------------------------------------------------------------------------------------------------------
# Launch geometry mirrors (the C++ they copy is cited; keep them in step with it)
# ------------------------------------------------------------------------------------------------------------------

def k6_geometry(R, Cout, groups):
    """conv_gemm.cu tile_width() (398-407) and launch_variant() (387-389): tile width, column tiles, tiles, grid."""
    bn = 256 if Cout > 128 else (128 if Cout > 64 else 64)
    if groups > 1:
        og = Cout // groups
        bn = next(c for c in (bn, 128, 64) if c <= bn and (og % c == 0 if og >= c else (c % og == 0 and og % 16 == 0)))
    col_tiles = -(-Cout // bn)
    tiles = -(-R // 128) * col_tiles
    return bn, col_tiles, tiles, min(tiles, _sms())


def assert_k6_walks(R, Cout, groups):
    """Every CTA takes >= 2 tiles (accumulator buffer 1, the tfull / tempty phase flips, moments carried across tiles)
    and the tile count is not a multiple of the grid (CTAs with different tile counts, an odd one among them)."""
    bn, col_tiles, tiles, grid = k6_geometry(R, Cout, groups)
    assert tiles // grid >= 2 and tiles % grid != 0, (R, Cout, groups, bn, tiles, grid)
    return bn, col_tiles, tiles, grid


def bn_geometry(R, C, V):
    """bn_fused.cu bn_geometry() (105-118): threads per row, rows per block pass, channel tiles, row blocks."""
    cv = C // V
    tpr = min(cv, 32)
    rpp = 256 // tpr
    ctiles = cv // tpr
    gx = min(-(-R // rpp), max(1, _sms() * 4 // ctiles))
    return tpr, rpp, ctiles, gx


def keep_rows_per_thread(mb, tensors, C, elem):
    """bn_fused.cu keep_rows_per_thread() (742-750): rows of pass 1 loaded "evict last", -1 = no cache hints."""
    if mb <= 0:
        return -1
    rows_kept = mb * 1048576.0 / (tensors * C * elem)
    rows_per_sweep = _sms() * 4 * 256 / (C / (16 // elem))
    k = rows_kept / rows_per_sweep
    return 0 if k < 1.0 else int(k)


def bn_persistent_rows(R, C, dtype, backward):
    """Rows per thread of the single-launch kernels (bn_fwd_t / bn_bwd_t try_launch: gx capped by the cooperative
    capacity; n = ceil((R - r0) / (gx * rpp)), bn_fused.cu 465 / 619) for every blocks-per-SM count the occupancy
    calculator may report: at least the kernel's __launch_bounds__ minimum (fwd fp32 4, fwd bf16 3, bwd 2), and beyond
    4 the grid no longer changes.  Returns [(blocks per SM, (fewest, most) rows per thread)]."""
    elem = 4 if dtype == torch.float32 else 2
    tpr, rpp, ctiles, gx = bn_geometry(R, C, 16 // elem)
    lo = 2 if backward else (4 if elem == 4 else 3)
    out = []
    for bps in range(lo, 5):
        g = min(gx, bps * _sms() // ctiles)
        step = g * rpp
        out.append((bps, (R // step, -(-R // step))))
    return out


def apply_items(R, C, dtype, per_sm):
    """(fewest, most) 16-byte items per thread of bn_apply_kernel (per_sm = 4) / bn_bwd_apply_kernel (8): apply_grid()
    (bn_fused.cu 752-760) and n = ceil((total - i0) / (grid * 256)) (257, 392)."""
    cv = C // (16 // (4 if dtype == torch.float32 else 2))
    total = R * cv
    g = min(_sms() * per_sm, -(-total // 256))
    q = cv // 256 if cv > 256 else 1
    g = -(-g // q) * q
    T = g * 256
    return total // T, -(-total // T)


def assert_rows_walk(n_lo, n_hi, keep=None):
    """n >= 8 rows per thread, threads with n and n - 1 rows (so both residues mod 4 of the unrolled loop's tail), and
    the evict-last split keep_from = n - keep strictly inside (0, n) for every thread."""
    assert n_lo >= 8 and n_hi == n_lo + 1, (n_lo, n_hi)
    if keep is not None:
        assert 1 <= keep < n_lo, (keep, n_lo)


def assert_bn_walks(R, C, dtype, keep_mb=80, persistent=True):
    elem = 4 if dtype == torch.float32 else 2
    if persistent:
        for backward, tensors in ((False, 1), (True, 2)):
            keep = keep_rows_per_thread(keep_mb, tensors, C, elem)
            for _, (lo, hi) in bn_persistent_rows(R, C, dtype, backward):
                assert_rows_walk(lo, hi, keep if keep >= 0 else None)
    else:
        for per_sm in (4, 8):
            assert_rows_walk(*apply_items(R, C, dtype, per_sm))
        tpr, rpp, ctiles, gx = bn_geometry(R, C, 16 // elem)      # the statistics / reduction kernels
        assert_rows_walk(R // (gx * rpp), -(-R // (gx * rpp)))


def knn_self_grid(N, B):
    """knn_tc2.cu plan_with() (904-913: the self kernel takes N <= 256, NH = 2 above 128 nodes) and launch_self()
    (862-863: one CTA per SM at NH = 2, two at NH = 1, at most B).  None: the streaming kernel (one CTA per query
    block and segment, nothing walks)."""
    if N > 256:
        return None
    return min(_sms() * (2 if N <= 128 else 1), B)


# ------------------------------------------------------------------------------------------------------------------
# Explicit tables of the shapes the step issues (checked against the step by test_step_shapes_are_all_covered)
# ------------------------------------------------------------------------------------------------------------------

# K6 (conv1x1_bn_stats_fwd): (N, Cin, Cout, groups) at B = 512.  The layers with more than 2 KB of k-range per row stay
# on cuDNN (ops.conv1x1_stats_ok): fp32 takes three fewer shapes than bf16.
K6_FP32 = [(1024, 64, 64, 1), (1024, 128, 128, 4), (1024, 128, 64, 1), (1024, 64, 256, 1), (1024, 256, 64, 1),
           (512, 192, 128, 1), (512, 128, 128, 1), (512, 256, 256, 4), (512, 256, 128, 1), (512, 128, 512, 1),
           (512, 512, 128, 1),
           (256, 384, 256, 1), (256, 256, 256, 1), (256, 512, 512, 4), (256, 512, 256, 1), (256, 256, 1024, 1),
           (128, 512, 512, 1), (128, 1024, 1024, 4), (128, 512, 2048, 1)]
K6_BF16 = K6_FP32 + [(256, 1024, 256, 1), (128, 1024, 512, 1), (128, 768, 512, 1)]
# synthetic: BN = 64 (one epilogue team per tile, alternating), 3 column tiles (flush on every tile), a ragged second
# column block, rows that are not a multiple of 128
K6_SYNTH = {"bn64": (512, 1024, 96, 64), "cout768": (512, 256, 256, 768), "cout384": (512, 256, 128, 384),
            "ragged_rows": (511, 1000, 64, 128)}
K6_CASES = ([pytest.param("fp32", B_STEP, *s, id=f"fp32-N{s[0]}-{s[1]}x{s[2]}g{s[3]}") for s in K6_FP32]
            + [pytest.param("bf16", B_STEP, *s, id=f"bf16-N{s[0]}-{s[1]}x{s[2]}g{s[3]}") for s in K6_BF16]
            + [pytest.param(dt, B, N, Cin, Cout, 1, id=f"{dt}-{name}") for name, (B, N, Cin, Cout) in K6_SYNTH.items()
               for dt in DTYPES])

# K5 (bn_train_fwd / bn_apply_fwd / bn_train_bwd): (B, N, C, mode).  A bf16 tensor of B = 512 rows with 64 channels
# per node (64 MB) fits the 80 MB evict-last budget whole (keep_from = 0): B = 768 there.
K5_STEP = {"fp32": [(512, 1024, 64, "plain"), (512, 1024, 128, "relu"), (512, 1024, 64, "residual"), (512, 1024, 256, "relu"),
                    (512, 512, 128, "plain"), (512, 512, 256, "relu"), (512, 512, 128, "residual"), (512, 512, 512, "relu"),
                    (512, 256, 256, "plain"), (512, 256, 512, "relu"), (512, 256, 256, "residual"), (512, 256, 1024, "relu"),
                    (512, 128, 512, "plain"), (512, 128, 1024, "relu"), (512, 128, 512, "residual"), (512, 128, 2048, "relu")]}
K5_STEP["bf16"] = [(768, 1024, 64, "plain"), (512, 1024, 128, "relu"), (768, 1024, 64, "residual"), (512, 1024, 256, "relu"),
                   (768, 512, 128, "plain"), (512, 512, 256, "relu"), (768, 512, 128, "residual"), (512, 512, 512, "relu"),
                   (768, 256, 256, "plain"), (512, 256, 512, "relu"), (768, 256, 256, "residual"), (512, 256, 1024, "relu"),
                   (768, 128, 512, "plain"), (512, 128, 1024, "relu"), (768, 128, 512, "residual"), (512, 128, 2048, "relu")]
K5_CASES = [pytest.param(dt, B, N, C, m, id=f"{dt}-B{B}-N{N}-C{C}-{m}") for dt, rows in K5_STEP.items() for B, N, C, m in rows]

# k-NN (knn_fwd) and K2 / K3 (mr_aggregate): every stage, k = 3.  At N = 128 the self kernel's grid is 2 * SMs: B = 600.
KNN_B = {1024: 512, 512: 512, 256: 512, 128: 600}
# tap rows (downsample_taps_fwd): the (N, C) input of each Downsample
TAPS = [(1024, 64), (512, 128), (256, 256)]


def _covers(name, meta):
    """Whether a (name, meta) the step issued is in the tables (everything but B must match)."""
    m = {k: v for k, v in meta.items() if k != "B"}
    dt = "fp32" if m.get("dtype", 0) == 0 else "bf16"
    if name == "conv1x1_bn_stats_fwd":
        table = K6_FP32 if dt == "fp32" else K6_BF16
        return (m["N"], m["Cin"], m["Cout"], m["groups"]) in table
    if name in ("bn_train_fwd", "bn_apply_fwd"):
        mode = "relu" if m["relu"] else ("residual" if m["res"] else "plain")
        return any((N, C, md) == (m["N"], m["C"], mode) for _, N, C, md in K5_STEP[dt])
    if name == "bn_train_bwd":
        return any((N, C) == (m["N"], m["C"]) and (md == "relu") == bool(m["relu"]) for _, N, C, md in K5_STEP[dt])
    if name == "knn_fwd":
        return (m["N"], m["C"]) in STAGES and m["M"] == m["N"] and m["K"] == 3
    if name == "mr_aggregate_fwd":
        return (m["N"], m["C"]) in STAGES and m["M"] == m["N"] and m["k"] == 3 and m["i64"] == 0
    if name == "downsample_taps_fwd":
        return (m["N"], m["C"]) in TAPS
    raise AssertionError(name)


_TRACKED = ("conv1x1_bn_stats_fwd", "bn_train_fwd", "bn_apply_fwd", "bn_train_bwd", "knn_fwd", "mr_aggregate_fwd",
            "downsample_taps_fwd")


@pytest.mark.parametrize("mode", ["fp32-tf32", "bf16-autocast"])
def test_step_shapes_are_all_covered(mode):
    """One train-mode forward + backward of the step's encoder at B = 512 (fp32 with TF32 convolutions and conv_gemm = 1,
    what bench.py runs, or under bf16 autocast): every shape it sends to the kernels under test appears in the tables
    of this module, so a model change that issues an untested shape fails here."""
    cfg = dict(synth.DEFAULT_CFG)
    torch.manual_seed(0)
    enc = GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3).to(DEV).train()
    n = cfg["n_mels"] * cfg["n_frames"] // cfg["peak_stride"]
    x = torch.relu(torch.randn(B_STEP, cfg["n_filters"], n, device=DEV, generator=_gen(1)))
    timer = ops.KernelTimer(timing=True)
    torch.backends.cudnn.allow_tf32 = True
    ops.set_timer(timer)
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "bf16-autocast"):
            out = enc(x)
        out.float().square().mean().backward()
    finally:
        ops.set_timer(None)
    torch.cuda.synchronize()
    seen = {(name, tuple(sorted(meta.items()))) for name, meta, _, _ in timer.records if name in _TRACKED}
    assert {name for name, _ in seen} == set(_TRACKED), seen
    missing = sorted((name, meta) for name, meta in seen if not _covers(name, dict(meta)))
    assert not missing, f"shapes of the step that no table of this module tests: {missing}"


# ------------------------------------------------------------------------------------------------------------------
# K6: conv1x1_stats_kernel (conv_gemm.cu)
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dt,B,N,Cin,Cout,groups", K6_CASES)
def test_conv1x1_stats_at_step_size(dt, B, N, Cin, Cout, groups):
    """y = x W^T and its per-channel moments with every CTA walking >= 2 tiles.

    Bound for y, element by element, with A = |X| |W|^T (fp64) and K = Cin (the dense k-range; a grouped schedule adds
    only exact zeros):
      * fp32 rows run as TF32: each operand keeps 10 mantissa bits, |dx / x|, |dw / w| <= u = 2^-10, so a product is
        off by <= (2u + u^2) |x w|; the fp32 accumulation of K products adds <= (K + 2) 2^-24 A (a chained sum of K
        terms: K - 1 roundings, 2 spare for the tensor core's own alignment); y is stored as accumulated:
        |y - y64| <= (2u + u^2 + (K + 2) 2^-24) A.
      * bf16 operands are exact in the product, the fp32 accumulation as above, then one rounding to bf16:
        |y - y64| <= 2^-8 |y64| + (1 + 2^-8) (K + 2) 2^-24 A.
    Moments: against double sums of the kernel's own output (fp32 partial sums over 64-row half tiles, the existing
    3e-6 bar), and against the fp64 sums of y64 within the summed element bound.  Batch invariance: a tile depends only
    on its rows and W, so rows computed in a call of their own must be bit-identical."""
    dtype = DTYPES[dt]
    R = B * N
    bn, col_tiles, tiles, grid = assert_k6_walks(R, Cout, groups)
    if Cout == 64:
        assert bn == 64 and any(t % 2 == 1 for t in (tiles // grid, tiles // grid + 1))   # team 1 takes odd lt only
    if Cout == 768:
        assert col_tiles == 3                                                                  # ct changes every tile
    lib = ops._native.load()
    assert lib.grafp_conv1x1_bn_stats_supported(R, Cin, Cout, groups, 0 if dtype == torch.float32 else 1) == 1
    g = _gen(R + Cin * 7 + Cout * 13 + groups)
    Cg = Cin // groups
    x = _cl((torch.randn(B, Cin, N, 1, device=DEV, generator=g) + 0.5).to(dtype))
    w = (torch.randn(Cout, Cg, 1, 1, device=DEV, generator=g) / Cg ** 0.5).to(dtype)
    h, ws = ops._conv1x1_stats_call(lib, x, w, groups)
    torch.cuda.synchronize()
    assert h.shape == (B, Cout, N, 1) and h.dtype == dtype and ops._is_rows(h)

    X = _rows(x).double()
    Wd = torch.block_diag(*w.double().reshape(groups, Cout // groups, Cg))             # (Cout, Cin)
    y64 = X @ Wd.T
    A = X.abs() @ Wd.abs().T
    y = _rows(h).double()
    acc = (Cin + 2) * U32
    bound = (2 * U_TF32 + U_TF32 ** 2 + acc) * A if dtype == torch.float32 else U_BF16 * y64.abs() + (1 + U_BF16) * acc * A
    err = (y - y64).abs()
    ratio = _ratio(err, bound)
    _note(f"K6 y {dt}", ratio)
    assert ratio <= 1.0, (ratio, int((err > bound).sum()))
    del X, A, err

    m = gio.bn_moments(ws, Cout)
    s1, s2 = y.sum(0), (y * y).sum(0)
    r2 = float((m[1] - s2).abs().max() / s2.abs().max()) / 3e-6
    bar1 = 1e-6 * float(s2.sum().sqrt()) * R ** 0.5 / Cout ** 0.5 + 1e-9
    r1 = float((m[0] - s1).abs().max()) / bar1
    _note("K6 moments vs own output", max(r1, r2))
    assert r1 <= 1.0 and r2 <= 1.0, (r1, r2)
    # against the fp64 GEMM: the moments of y64 move by at most the summed element bound
    sb = bound.sum(0)
    r3 = _ratio((m[0] - y64.sum(0)).abs(), sb + bar1)
    r4 = _ratio((m[1] - (y64 * y64).sum(0)).abs(), (2 * y64.abs() * bound + bound * bound).sum(0) + 3e-6 * s2.abs().max())
    _note("K6 moments vs fp64", max(r3, r4))
    assert r3 <= 1.0 and r4 <= 1.0, (r3, r4)
    del y64, bound

    # batch invariance: the first segments, ones in the middle of the walk, the last ones
    for b0, b1 in ((0, 1), (B // 2 - 1, B // 2 + 2), (B - 2, B)):
        hs, _ = ops._conv1x1_stats_call(lib, _cl(x[b0:b1]), w, groups)
        assert torch.equal(hs, h[b0:b1]), (b0, b1)


# ------------------------------------------------------------------------------------------------------------------
# K5: fused train-mode BatchNorm (bn_fused.cu)
# ------------------------------------------------------------------------------------------------------------------

def _bn_inputs(B, N, C, dtype, seed):
    g = _gen(seed)
    std = 0.5 + 2.5 * torch.rand(1, C, 1, 1, device=DEV, generator=g)
    x = (torch.randn(B, C, N, 1, device=DEV, generator=g) * std + 40.0 * torch.randn(1, C, 1, 1, device=DEV, generator=g))
    res = torch.randn(B, C, N, 1, device=DEV, generator=g)
    up = torch.randn(B, C, N, 1, device=DEV, generator=g)
    bn_ref = torch.nn.BatchNorm2d(C).double().to(DEV)
    with torch.no_grad():
        bn_ref.weight.copy_(torch.randn(C, device=DEV, generator=g).double())
        bn_ref.bias.copy_(torch.randn(C, device=DEV, generator=g).double())
        bn_ref.running_mean.copy_(torch.randn(C, device=DEV, generator=g).double())
        bn_ref.running_var.copy_(torch.rand(C, device=DEV, generator=g).double() + 0.5)
    return _cl(x.to(dtype)), _cl(res.to(dtype)), _cl(up.to(dtype)), bn_ref


def _float_copy(bn_ref):
    bn = torch.nn.BatchNorm2d(bn_ref.num_features).to(DEV)
    bn.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in bn_ref.state_dict().items()})
    return bn.train()


def _bn_bounds(x64, bn_ref, n_rows):
    """Per-channel error bounds of the fused BatchNorm in fp32 arithmetic (u = 2^-24), from the fp64 data.

    Statistics: each thread sums (x - s) and (x - s)^2 about s = row 0 in fp32 over <= n rows, then a tree over <= 256
    lanes: relative error <= e = (n + 8) u of the sums of magnitudes.  So the mean is off by
    dmu <= e mean|x - s| + 2 u |mu| (the float conversion), the variance by dvar <= e (mean (x - s)^2 + 2 |mu - s|
    mean|x - s|), and the float invstd / a = gamma invstd by eps_is <= dvar / (2 (var + eps)) + 3 u.
    Forward, with M = max|xhat|: |y - y64| <= |gamma| invstd (dmu + u max|x - mu|) + |gamma| M (eps_is + u)
    + u (|gamma| M + |beta|)  (+ u max|y + residual| for the residual add).  With the per-channel offsets of 40 sigma the
    dmu term (the mean rounded to fp32 before the subtraction) is the large one: the scale is |gamma| max|xhat| + |beta|
    plus |gamma| |mu| / sigma.
    Returns a dict of per-channel tensors used by the forward and backward checks."""
    C = x64.shape[1]
    X = _rows(x64)
    e = (n_rows + 8) * U32
    mu = X.mean(0)
    var = X.var(0, unbiased=False)
    s = X[0]
    dev = (X - s).abs().mean(0)
    dmu = e * dev + 2 * U32 * mu.abs()
    dvar = e * ((X - s).square().mean(0) + 2 * (mu - s).abs() * dev)
    eps_is = dvar / (2 * (var + bn_ref.eps)) + 3 * U32
    invstd = (var + bn_ref.eps).rsqrt()
    D = (X - mu).abs().amax(0)
    M = D * invstd
    gam, bet = bn_ref.weight.detach().abs(), bn_ref.bias.detach().abs()
    fwd = gam * invstd * (dmu + U32 * D) + gam * M * (eps_is + U32) + U32 * (gam * M + bet)
    dxhat = invstd * dmu + M * eps_is + 2 * U32 * M
    return dict(e=e, fwd=fwd.view(1, C), M=M, invstd=invstd, eps_is=eps_is, dxhat=dxhat, gam=gam)


def _check_bn_forward(got, pre64, ref64, b, dtype, relu, residual, family):
    """got vs ref64 element by element within the per-channel bound (+ the bf16 rounding of the stored output)."""
    G = _rows(got.detach()).double()
    Rf = _rows(ref64.detach())
    bound = b["fwd"].clone()
    if residual is not None:
        bound = bound + U32 * Rf.abs().amax(0, keepdim=True)
    bound = bound + (U_BF16 * Rf.abs() if dtype == torch.bfloat16 else 0.0)
    ratio = _ratio((G - Rf).abs(), bound)
    _note(family, ratio)
    assert ratio <= 1.0, ratio
    if relu:  # the mask may differ from fp64 only where the fp64 pre-activation is within the bound of zero
        P = _rows(pre64.detach())
        flip = (G > 0) != (P > 0)
        assert bool((P[flip].abs() <= (b["fwd"].expand_as(P)[flip] + 1e-30)).all())


def _check_bn_backward(dx, dw, db, x64, up64, mask, bn_ref, b, dtype, family):
    """dx, dgamma, dbeta against the fp64 gradients of the same masked output (the kernel's own ReLU mask).

    With gz = dy masked, c1 = mean gz, c2 = mean gz xhat and a = gamma invstd, dx = a (gz - c1 - xhat c2).  The kernel's
    mean / invstd carry the forward's errors (dxhat <= invstd dmu + M eps_is + 2 u M); its sums add e = (n + 8) u:
    dc1 <= e mean|gz|, dc2 <= e mean|gz xhat| + mean|gz| dxhat, so per channel
    |dx - dx64| <= |a| ((eps_is + 5 u)(max|gz| + |c1| + M |c2|) + dc1 + M dc2 + |c2| dxhat)  (+ 2^-8 |dx64| in bf16),
    |dbeta - dbeta64| <= e sum|gz| + u |dbeta|, |dgamma - dgamma64| <= e sum|gz xhat| + sum|gz| dxhat + u |dgamma|."""
    X = _rows(x64)
    gz = _rows(up64) * _rows(mask)
    mu, invstd = X.mean(0), b["invstd"]
    xhat = (X - mu) * invstd
    c1, c2 = gz.mean(0), (gz * xhat).mean(0)
    a = bn_ref.weight.detach() * invstd
    M, e, eps_is, dxhat = b["M"], b["e"], b["eps_is"], b["dxhat"]
    dc1 = e * gz.abs().mean(0)
    dc2 = e * (gz * xhat).abs().mean(0) + gz.abs().mean(0) * dxhat
    scale = gz.abs().amax(0) + c1.abs() + M * c2.abs()
    bdx = a.abs() * ((eps_is + 5 * U32) * scale + dc1 + M * dc2 + c2.abs() * dxhat)
    dx64 = a * (gz - c1 - xhat * c2)
    bound = bdx.view(1, -1) + (U_BF16 * dx64.abs() if dtype == torch.bfloat16 else 0.0)
    r_dx = _ratio((_rows(dx).double() - dx64).abs(), bound)
    s1, s2 = gz.sum(0), (gz * xhat).sum(0)
    r_db = _ratio((db.double() - s1).abs(), e * gz.abs().sum(0) + U32 * s1.abs())
    r_dw = _ratio((dw.double() - s2).abs(), e * (gz * xhat).abs().sum(0) + gz.abs().sum(0) * dxhat + U32 * s2.abs())
    _note(family, max(r_dx, r_db, r_dw))
    assert r_dx <= 1.0 and r_db <= 1.0 and r_dw <= 1.0, (r_dx, r_db, r_dw)


def _run_bn(dt, B, N, C, mode, seed):
    """Two train-mode steps through ops.batch_norm_act against nn.BatchNorm2d in fp64 on the GPU, then the backward."""
    dtype = DTYPES[dt]
    xg, rg, up, bn_ref = _bn_inputs(B, N, C, dtype, seed)
    bn = _float_copy(bn_ref)
    bn_ref.train()
    xg.requires_grad_(True)
    rg.requires_grad_(True)
    x64 = xg.detach().double().requires_grad_(True)
    r64 = rg.detach().double()
    relu, residual = mode == "relu", (rg if mode == "residual" else None)
    for _ in range(2):  # the running statistics accumulate over two steps
        got = ops.batch_norm_act(xg, bn, relu=relu, residual=residual)
        pre64 = bn_ref(x64) + (r64 if residual is not None else 0.0)
    ref64 = torch.relu(pre64) if relu else pre64
    assert got.dtype == dtype and ops._is_rows(got)
    assert int(bn.num_batches_tracked) == int(bn_ref.num_batches_tracked) == 2
    # the existing norm bars
    assert gio.rel_err(got, ref64) < (2e-5 if dtype == torch.float32 else 4e-3)
    assert gio.rel_err(bn.running_mean, bn_ref.running_mean) < 1e-5
    assert gio.rel_err(bn.running_var, bn_ref.running_var) < 1e-5
    _, (n_lo, n_hi) = bn_persistent_rows(B * N, C, dtype, False)[0]
    n_rows = max(n_hi * 2, max(apply_items(B * N, C, dtype, 4)))      # (<= the smallest grid the occupancy allows)
    bnd = _bn_bounds(x64.detach(), bn_ref, n_rows)
    _check_bn_forward(got, pre64, ref64, bnd, dtype, relu, residual, f"K5 fwd {dt}")
    mask = (got.detach() > 0).double() if relu else torch.ones_like(x64)
    got.backward(up)
    (pre64 * mask).backward(up.double())
    assert gio.rel_err(xg.grad, x64.grad) < (1e-4 if dtype == torch.float32 else 1e-2)
    assert gio.rel_err(bn.weight.grad, bn_ref.weight.grad) < (1e-4 if dtype == torch.float32 else 2e-3)
    assert gio.rel_err(bn.bias.grad, bn_ref.bias.grad) < (1e-4 if dtype == torch.float32 else 2e-3)
    if residual is not None:
        assert torch.equal(rg.grad, up)
    _check_bn_backward(xg.grad, bn.weight.grad, bn.bias.grad, x64.detach(), up.double(), mask, bn_ref, bnd, dtype,
                       f"K5 bwd {dt}")


@pytest.mark.parametrize("dt,B,N,C,mode", K5_CASES)
def test_batch_norm_at_step_size(dt, B, N, C, mode):
    """Every (rows, channels, ReLU / residual, dtype) BatchNorm of the step through ops.batch_norm_act, forward and
    backward, at default options (the single-launch kernels), with large per-channel offsets (40 sigma)."""
    assert_bn_walks(B * N, C, DTYPES[dt])
    _run_bn(dt, B, N, C, mode, seed=B * 7 + N + C)


def _near_end_keep_mb(C, elem):
    """bn_l2_keep_mb that makes keep_rows_per_thread() 1 in the backward (two tensors) and 2 in the forward: the
    evict-last split sits one or two rows before the end of every thread's walk."""
    sweep_bytes = _sms() * 4 * 256 / (C / (16 // elem)) * C * elem
    return math.ceil(2 * sweep_bytes / 1048576.0)


BN_SWEEP_SHAPE = {"fp32": (512, 1024, 64, "residual"), "bf16": (512, 1024, 128, "relu")}
BN_OPTION_SETS = ([(1, rev, keep) for rev in (1, 0) for keep in (0, 80, "near-end")] + [(0, rev, 80) for rev in (1, 0)])


@pytest.mark.parametrize("persistent,reverse,keep_mb", BN_OPTION_SETS)
@pytest.mark.parametrize("dt", ["fp32", "bf16"])
def test_batch_norm_loop_copies_at_step_size(dt, persistent, reverse, keep_mb):
    """The separately compiled loop copies of K5 on one stage-0 shape per dtype: the single launch with and without L2
    hints and with the evict-last split near the end of the walk, first pass reversed or not, and the two-kernel pair
    (statistics / reduction + bn_apply_kernel / bn_bwd_apply_kernel)."""
    B, N, C, mode = BN_SWEEP_SHAPE[dt]
    dtype = DTYPES[dt]
    elem = 4 if dtype == torch.float32 else 2
    mb = _near_end_keep_mb(C, elem) if keep_mb == "near-end" else keep_mb
    if keep_mb == "near-end":
        assert keep_rows_per_thread(mb, 2, C, elem) == 1 and keep_rows_per_thread(mb, 1, C, elem) == 2
    if persistent:
        for backward, tensors in ((False, 1), (True, 2)):
            keep = keep_rows_per_thread(mb, tensors, C, elem)
            for _, (lo, hi) in bn_persistent_rows(B * N, C, dtype, backward):
                assert_rows_walk(lo, hi, keep if keep >= 0 else None)
    else:
        assert_bn_walks(B * N, C, dtype, persistent=False)
    ops.set_option("bn_persistent", persistent)
    ops.set_option("bn_reverse", reverse)
    ops.set_option("bn_l2_keep_mb", mb)
    _run_bn(dt, B, N, C, mode, seed=11 + persistent * 2 + reverse)


STAGE0_CONV_BN = [(64, 64, 1, "plain", True), (128, 128, 4, "relu", True), (128, 64, 1, "residual", True),
                  (64, 256, 1, "relu", False), (256, 64, 1, "residual", False)]


@pytest.mark.parametrize("Cin,Cout,groups,mode,bias", STAGE0_CONV_BN,
                         ids=[f"{a}x{b}g{g}-{m}" for a, b, g, m, _ in STAGE0_CONV_BN])
def test_conv_batch_norm_from_moments_at_step_size(Cin, Cout, groups, mode, bias):
    """The apply-from-moments path end to end (K6 GEMM + statistics epilogue, bn_apply_kernel, the fused backward with
    the convolution-bias gradient from dx_colsum) at the stage-0 layers of the step, TF32 allowed and conv_gemm = 1,
    against Conv2d + BatchNorm2d in fp64.

    Bounds: h carries the K6 element bound Bh = (2u + u^2 + (K + 2) 2^-24) |X||W|^T (u = 2^-10); the BatchNorm maps
    it through gamma invstd, and its mean / variance through the same factor, so per channel
    |out - out64| <= |gamma| invstd (max Bh + mean Bh + M mean(Bh |xhat|)) + the fp32 apply bound of _bn_bounds
    (n = 64 rows per partial sum).  Running statistics and gradients: the TF32 norm bar 3e-3 of the existing GEMM-path
    test (TF32 truncation biases the mean and the variance by ~2^-11), dbeta 1e-4 (no TF32 in it).  The bias gradient is
    analytically zero; the kernel's is the rounding residue a (s1 - R fl(s1 / R)) - a invstd c2 s3, s3 = sum (h - mu)
    in fp32 over <= ~120 rows per thread about the fp32 mean of the epilogue's 64-row partial sums:
    |dbias_c| <= 2^-15 |a| (sum|gz| + |c2| (sum|xhat| + R |mu| invstd))."""
    B, N = B_STEP, 1024
    R = B * N
    assert_k6_walks(R, Cout, groups)
    for per_sm in (4, 8):
        assert_rows_walk(*apply_items(R, Cout, torch.float32, per_sm))
    g = _gen(Cin * 3 + Cout + groups)
    conv_ref = torch.nn.Conv2d(Cin, Cout, 1, groups=groups, bias=bias).double().to(DEV)
    bn_ref = torch.nn.BatchNorm2d(Cout).double().to(DEV).train()
    with torch.no_grad():
        conv_ref.weight.copy_(torch.randn(conv_ref.weight.shape, device=DEV, generator=g).double() / (Cin // groups) ** 0.5)
        if bias:
            conv_ref.bias.copy_(torch.randn(Cout, device=DEV, generator=g).double())
        bn_ref.weight.copy_(torch.randn(Cout, device=DEV, generator=g).double())
        bn_ref.bias.copy_(torch.randn(Cout, device=DEV, generator=g).double())
    conv = torch.nn.Conv2d(Cin, Cout, 1, groups=groups, bias=bias).to(DEV)
    conv.load_state_dict({k: v.float() for k, v in conv_ref.state_dict().items()})
    bn = _float_copy(bn_ref)
    x = _cl(torch.randn(B, Cin, N, 1, device=DEV, generator=g) + 0.5)
    res = _cl(torch.randn(B, Cout, N, 1, device=DEV, generator=g))
    up = _cl(torch.randn(B, Cout, N, 1, device=DEV, generator=g))
    xg = x.clone().requires_grad_(True)
    x64 = x.double().requires_grad_(True)
    torch.backends.cudnn.allow_tf32 = True
    timer = ops.KernelTimer(timing=True)
    ops.set_timer(timer)
    try:
        got = ops.conv_batch_norm_act(xg, conv, bn, relu=mode == "relu", residual=res if mode == "residual" else None)
    finally:
        ops.set_timer(None)
    assert [rec[0] for rec in timer.records] == ["conv1x1_bn_stats_fwd", "bn_apply_fwd"]
    h64 = conv_ref(x64)
    pre64 = bn_ref(h64) + (res.double() if mode == "residual" else 0.0)
    ref64 = torch.relu(pre64) if mode == "relu" else pre64

    with torch.no_grad():
        X = _rows(x).double()
        Wd = torch.block_diag(*conv_ref.weight.abs().reshape(groups, Cout // groups, Cin // groups))
        Bh = (2 * U_TF32 + U_TF32 ** 2 + (Cin + 2) * U32) * (X.abs() @ Wd.T)
        del X
        h_nobias = h64.detach() - conv_ref.bias.detach().view(1, -1, 1, 1) if bias else h64.detach()
        b = _bn_bounds(h_nobias, bn_ref, 64)
        H = _rows(h64.detach())
        xhat = (H - H.mean(0)) * b["invstd"]
        tf = b["gam"] * b["invstd"] * (Bh.amax(0) + Bh.mean(0) + b["M"] * (Bh * xhat.abs()).mean(0))
        b["fwd"] = b["fwd"] + tf.view(1, -1)
        del Bh, H
        _check_bn_forward(got, pre64, ref64, b, torch.float32, mode == "relu", res if mode == "residual" else None,
                          "K6+K5 apply-from-moments fwd")
    assert int(bn.num_batches_tracked) == 1
    assert gio.rel_err(bn.running_var, bn_ref.running_var) < 3e-3
    assert gio.rel_err(bn.running_mean, bn_ref.running_mean) < 3e-3

    mask = (got.detach() > 0).double() if mode == "relu" else torch.ones_like(ref64)
    got.backward(up)
    (pre64 * mask).backward(up.double())
    for mine, ref in ((xg.grad, x64.grad), (conv.weight.grad, conv_ref.weight.grad), (bn.weight.grad, bn_ref.weight.grad)):
        assert gio.rel_err(mine, ref) < 3e-3
    assert gio.rel_err(bn.bias.grad, bn_ref.bias.grad) < 1e-4     # the sum of the masked gradient: no TF32 in it
    if bias:
        gz = _rows(up.double() * mask)
        c2 = (gz * xhat).mean(0)
        a = b["gam"] * b["invstd"]
        mu = _rows(h64.detach()).mean(0) - conv_ref.bias.detach()       # the kernel's h has no bias
        lim = 2.0 ** -15 * a * (gz.abs().sum(0) + c2.abs() * (xhat.abs().sum(0) + R * mu.abs() * b["invstd"]))
        ratio = _ratio(conv.bias.grad.double().abs(), lim)
        _note("K5 conv-bias gradient (dx colsum)", ratio)
        assert ratio <= 1.0, ratio


# ------------------------------------------------------------------------------------------------------------------
# K1: knn_self_kernel (knn_tc2.cu) and the streaming kernel at the step's shapes
# ------------------------------------------------------------------------------------------------------------------

def _planted_segments(grid, B):
    """Segments that come second or later in a CTA's walk of the self kernel (b >= grid), spread over the walk."""
    return sorted({grid + 1, grid + 4, 2 * grid + 1, B - 1} & set(range(grid, B)))


def _knn_input(B, N, C, dtype, planted):
    """ReLU'd N(0, 1) features.  In each planted segment one all-zero node (at a different index per segment, so that
    no two segments of a walk share the zero node's position) and one duplicated node: those segments' key norms are
    not all 1, so they take the vote-gated scan while the others of the same walk take the group maxima."""
    x = torch.relu(torch.randn(B, C, N, 1, device=DEV, generator=_gen(N * 31 + C)))
    for i, b in enumerate(planted):
        z = (17 + 37 * i) % N
        x[b, :, z] = 0
        x[b, :, (z + 5) % N] = x[b, :, (z + 9) % N]
    return _cl(x.to(dtype))


@pytest.mark.parametrize("dt", ["fp32", "bf16"])
@pytest.mark.parametrize("N,C", STAGES)
def test_knn_at_step_size(N, C, dt):
    """Every segment's graph against the fp64 distance ranking (O.knn_mismatch_report on the GPU, in chunks): no hard
    mismatch, and at most 2 % tie-order differences.  Batch invariance: a segment's graph alone equals its graph
    inside the full call (planted segments and a few others)."""
    dtype = DTYPES[dt]
    B, k = KNN_B[N], 3
    grid = knn_self_grid(N, B)
    if grid is not None:
        assert B >= 2 * grid, (B, grid)        # every CTA walks >= 2 segments: the TMA ring crosses a segment boundary
        planted = _planted_segments(grid, B)
        assert len(planted) >= 3 and min(planted) >= grid
    else:
        planted = [149, 297, 300, B - 1]
    x = _knn_input(B, N, C, dtype, planted)
    nn_idx, nn32 = ops.knn_graph(x, k)
    assert ops.knn_last_algo() == "tcgen05" and ops.knn_last_variant() == "f16x3"
    assert torch.equal(nn_idx, nn32.long())
    xf = x.float()   # bf16: the kernel normalises the bf16 values; the reference ranks the same values in fp64
    chunk = max(1, (1 << 25) // (N * N))
    for b0 in range(0, B, chunk):
        rep = O.knn_mismatch_report(xf[b0:b0 + chunk], nn_idx[b0:b0 + chunk], k, ordered=True)
        assert rep["hard"] == 0, (b0, rep)
        assert rep["mismatch"] <= 0.02 * rep["entries"], (b0, rep)
        _note(f"k-NN tie-order differences / 2% ({dt})", rep["mismatch"] / (0.02 * rep["entries"]))
    for b in sorted(set(planted) | {0, 1, B // 2}):
        alone, _ = ops.knn_graph(_cl(x[b:b + 1]), k)
        assert torch.equal(alone[0], nn_idx[b]), b
    if grid is not None:
        # with 256 or more channels the zero node (distance 1) is nearer than almost every other node (2 - 2 cos, cos of
        # two ReLU'd Gaussian rows ~ 1 / pi): a hub of its segment, so its key norm decides much of the segment's graph
        for i, b in enumerate(planted):
            z = (17 + 37 * i) % N
            assert int((nn_idx[b, :, 1:] == z).sum()) > N // 8, b


# ------------------------------------------------------------------------------------------------------------------
# K2 / K3 (aggregate.cu) and the tap rows (downsample.cu)
# ------------------------------------------------------------------------------------------------------------------

def _mr_reference(x, nbr):
    """Gather + max over the k neighbours in the input dtype (x_j - x_i rounded like the dtype, first maximiser), on the
    GPU.  Returns the interleaved output and the winning slot per (b, n, c)."""
    X = _rows(x).view(x.shape[0], x.shape[2], x.shape[1])                       # (B, N, C)
    bidx = torch.arange(x.shape[0], device=DEV).view(-1, 1, 1)
    xj = X[bidx, nbr.long()]                                                   # (B, N, k, C)
    d = (xj - X.unsqueeze(2)).to(x.dtype)
    best = d.max(2).values
    k = nbr.shape[-1]
    slot = torch.where(d == best.unsqueeze(2), torch.arange(k, device=DEV).view(1, 1, k, 1), k).amin(2)
    out = torch.stack([X, best], dim=-1).reshape(x.shape[0], x.shape[2], 2 * x.shape[1])
    return out, slot


def _mr_grad_reference(g, nbr, slot, B, N, C):
    """dx in fp64 by index_add_: dx_i = g_even_i - g_odd_i + the g_odd_n of every (n, c) whose winning neighbour is i
    (a node that wins its own row gets its g_odd back); plus, per element, the number of scattered terms and the fp64
    sum of the magnitudes of all its terms."""
    G = _rows(g).double().view(B, N, C, 2)
    ge, go = G[..., 0], G[..., 1]
    j = slot.long().view(B, N, C)                                                # winning slot per (b, n, c)
    target = torch.gather(nbr.long().unsqueeze(-1).expand(B, N, nbr.shape[-1], C), 2, j.unsqueeze(2)).squeeze(2)
    flat = ((target + torch.arange(B, device=DEV).view(B, 1, 1) * N) * C + torch.arange(C, device=DEV).view(1, 1, C)).view(-1)
    dx = (ge - go).reshape(-1).index_add_(0, flat, go.reshape(-1))
    mag = (ge.abs() + go.abs()).reshape(-1).index_add_(0, flat, go.abs().reshape(-1))
    terms = torch.zeros(B * N * C, device=DEV, dtype=torch.float64).index_add_(0, flat, torch.ones_like(go).reshape(-1))
    return dx.view(B, N, C), mag.view(B, N, C), terms.view(B, N, C)


@pytest.mark.parametrize("dt", ["fp32", "bf16"])
@pytest.mark.parametrize("N,C", STAGES)
def test_mr_aggregate_at_step_size(N, C, dt):
    """K2 forward bit for bit against a GPU gather + max; the K3 backward forms (fp32: 2, 1, 0 and the deterministic
    gather form 3; bf16: 2 and 0) against an fp64 index_add_, element by element: a sum of (in-degree + 2) terms in
    any order is within (in-degree + 1) u sum|terms| of the exact sum (u = 2^-24, or 2^-8 with bf16 accumulation
    and output; a single rounding can reach this bound, so ratios close to 1 are expected).  The graph is the k-NN
    graph of ReLU'd features with a hub: node 5 of every segment holds 2.0 in every channel and the last slot of every
    other row points at it, so x_5 - x_i wins most channels of those rows and node 5 collects ~N / 2 terms each."""
    dtype = DTYPES[dt]
    B, k = B_STEP, 3
    x = torch.relu(torch.randn(B, C, N, 1, device=DEV, generator=_gen(N + C)))
    x[:, :, 5] = 2.0
    x = _cl(x.to(dtype))
    _, nbr32 = ops.knn_graph(x, k)
    nbr32[:, 1::2, k - 1] = 5
    up = _cl(torch.randn(B, 2 * C, N, 1, device=DEV, generator=_gen(3)).to(dtype))
    ref, slot = _mr_reference(x, nbr32)
    dx64, mag, terms = _mr_grad_reference(up, nbr32, slot, B, N, C)
    u = U32 if dtype == torch.float32 else U_BF16
    assert float(terms[:, 5].mean()) > N / 4                                   # the hub
    bound = (terms + 1) * u * mag
    for form in ((2, 1, 0, 3) if dtype == torch.float32 else (2, 0)):
        ops.set_option("mr_bwd_form", form)
        xg = x.clone().requires_grad_(True)
        out = ops.mr_aggregate(xg, nbr32)
        assert torch.equal(_rows(out.detach()).view(B, N, 2 * C), ref), form
        (gx,) = torch.autograd.grad(out, xg, up)
        err = (_rows(gx).double().view(B, N, C) - dx64).abs()
        ratio = _ratio(err, bound)
        _note(f"K3 backward {dt}", ratio)
        assert ratio <= 1.0, (form, ratio)


@pytest.mark.parametrize("dt", ["fp32", "bf16"])
@pytest.mark.parametrize("N,C", TAPS)
def test_downsample_taps_at_step_size(N, C, dt):
    """Tap rows (x[2n'-1], x[2n'], x[2n'+1]) forward and backward at the step's Downsample inputs, bit-exact against the
    PyTorch construction of the same rows (pad + slice + cat) and its autograd."""
    dtype = DTYPES[dt]
    B = B_STEP
    g = _gen(N + C)
    x0 = _cl(torch.randn(B, C, N, 1, device=DEV, generator=g).to(dtype))
    up = _cl(torch.randn(B, 3 * C, N // 2, 1, device=DEV, generator=g).to(dtype))
    x = x0.clone().requires_grad_(True)
    taps = ops._DownsampleTaps.apply(x)
    taps.backward(up)
    xr = x0.clone().requires_grad_(True)
    rows = xr.permute(0, 2, 3, 1).reshape(B, N // 2, 2 * C)
    prev = torch.nn.functional.pad(rows[:, :-1, C:], (0, 0, 1, 0))
    ref = torch.cat([prev, rows], dim=2).view(B, N // 2, 1, 3 * C).permute(0, 3, 1, 2)
    ref.backward(up)
    assert taps.shape == ref.shape and torch.equal(taps, ref)
    assert torch.equal(x.grad, xr.grad)
