"""The dense part of a DLRM-Criteo training step against float64, at the bench batch and at the tile edges of its kernels.

Every comparison is |got - ref| <= bound, with ref computed in float64 from the same fp32 inputs and weights, and the
bound an error model in units of U = 2^-23 (one fp32 ulp at 1; the tensor cores truncate their accumulator, so a rounding
costs up to a whole ulp):

    |got - ref| <= c * U * (|A| @ |B|)

|A| @ |B| is taken in float64 over absolute values, so cancellation cannot hide an error.  c counts the roundings a term
can go through on its way into the result: the additions of the summation (its length, or for the row-direction sums of
the backward pass the length of the longest serial chain of the kernel's reduction) plus, for the 3xTF32 split,

    x = hi + lo + r,  hi = rna_tf32(x), |x - hi| <= 2^-11 |x|, lo = rna_tf32(x - hi), |r| <= 2^-22 |x|
    x * w - (hi_x hi_w + hi_x lo_w + lo_x hi_w) = lo_x lo_w + hi_x r_w + r_x hi_w + ...  ->  <= 3 * 2^-22 = 6 U

The whole step (section 1) carries the same model through the network: every quantity travels with its bound, and a
layer's bound is what its inputs' bounds become through it plus its own c * U * (|A| @ |B|) term.
"""
import itertools
import math
from collections import Counter

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0 ** -23
SPLIT = 6             # 3xTF32: the dropped lo*lo term and the two representation errors, 2^-22 each (docstring)
SMS = 148


# ---- error-model helpers ------------------------------------------------------------------------------------------------
def _mm(a, ea, b, eb, c, add=None, e_add=None):
    """a @ b (+ add) in float64 and a bound on how far a kernel that sums the products with c roundings per term can be
    from it when its operands are off by up to ea, eb:  |a| eb + ea (|b| + eb)  (propagated)  +  c U (|a| + ea)(|b| + eb)
    (its own roundings; `add` counts as one more term)."""
    y = a @ b
    aa, ab = a.abs(), b.abs()
    own = (aa + ea) @ (ab + eb)
    e = aa @ eb + ea @ (ab + eb)
    if add is not None:
        y = y + add
        own = own + add.abs() + e_add
        e = e + e_add
    return y, e + c * U * own


def _check(name, got, ref, bound):
    got = got.detach().double().reshape(ref.shape)
    err = (got - ref).abs()
    ok = err <= bound                                   # NaN fails
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        ratio = float(torch.nan_to_num(err / bound.clamp_min(1e-300), nan=math.inf).max())
        raise AssertionError(f"{name}: {bad.shape[0]} of {ref.numel()} elements outside the bound (worst err/bound "
                             f"{ratio:.3g}); first at {i}: got {float(got[i])!r}, float64 {float(ref[i])!r}, "
                             f"bound {float(bound[i]):.3g}")


def _kernels_run(fn):
    """fn() under torch.profiler -> (its result, the names of the CUDA kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # the first kernels after the profiler starts are not always recorded: these absorb that
        torch.ones(1, device=DEV).add_(1)
        torch.cuda.synchronize()
        out = fn()
        torch.cuda.synchronize()
    return out, " | ".join(sorted({e.name for e in prof.events() if e.device_type.name == "CUDA"}))


def _rows_c(M):
    """Longest serial chain of the row-direction sums of the hand-written backward kernels (dW, db of the narrow layers,
    the fused tail's sums, act_bwd_colsum, the BCE loss): a CTA adds its R rows one after another (a row-group fold
    at most doubles that), then the reduction kernel adds the G CTA partials in 8 interleaved chains plus an 8-way fold."""
    dw_g = min(max(-(-M // 32), 1), SMS * 4)                            # tzk_bwd2::dw_grid
    tail_g = min(max(-(-M // 128), 1), SMS * 4)                         # tzk_tail::grid_for
    tail_r = -(-(-(-M // tail_g)) // 128) * 128
    return max(2 * -(-M // dw_g) + dw_g, tail_r + tail_g, 128 + -(-M // 128)) + 16


def _wgrad3x_c(M, slabs):
    """tzk_wgrad3x: one accumulator per work item takes at most slab_rows terms, the epilogue adds 8 accumulators, the
    reduce kernel adds the `used` slabs in order; + SPLIT."""
    slab_rows = -(-(-(-M // slabs)) // 32) * 32
    used = -(-M // slab_rows)
    return slab_rows + used + 8 + SPLIT + 2


def _gemm3x_c(K):
    """tzk_gemm3x: an accumulator takes at most K terms (K padded with zeros to a multiple of 32 adds nothing), the
    epilogue adds <= 4 partial accumulators and the bias; + SPLIT."""
    return K + 5 + SPLIT + 2


# ---- inputs ---------------------------------------------------------------------------------------------------------------
def _ties(g, shape, generic=0.125):
    """Positive values on TF32 rounding ties, (m + 1/2) 2^(e - 10) with m in [1024, 2048): the 13 bits tf32 drops are
    exactly 1000...0, so rna rounds away and lo = -1/2 TF32 ulp, the largest lo there is, with the same sign for every
    element — dropping a lo term then shifts the result by ~2^-11.5 of |A| @ |B|, far outside the bounds below.
    A fraction `generic` of the elements are ordinary values."""
    d = g.device
    m = torch.randint(1024, 2048, shape, generator=g, device=d).double()
    e = torch.randint(-2, 3, shape, generator=g, device=d).double()
    v = (m + 0.5) * torch.exp2(e - 10)
    other = torch.rand(shape, generator=g, device=d).double() + 0.5
    return torch.where(torch.rand(shape, generator=g, device=d) < generic, other, v).float()


def _row_scaled(g, rows, cols, sign=None, scale=None):
    """_ties rows with a sign and a power-of-two scale per row (2^-10 .. 2^10, ~1e-3 .. 1e3; powers of two keep the ties)."""
    d = g.device
    if sign is None:
        sign = torch.where(torch.rand(rows, 1, generator=g, device=d) < 0.5, -1.0, 1.0)
    if scale is None:
        scale = torch.exp2(torch.randint(-10, 11, (rows, 1), generator=g, device=d).float())
    return (_ties(g, (rows, cols)) * sign * scale), sign, scale


# ==========================================================================================================================
# 2. tcgen05 GEMM passes (csrc/tzk_gemm3x.cu) at their edges
# ==========================================================================================================================
GEMM_M = [1, 31, 32, 127, 128, 129, 256, 384, SMS * 128, SMS * 128 + 1, 65536, 131072 + 3]
GEMM_K = [112, 224, 448, 784, 896]


@pytest.mark.parametrize("Kx", GEMM_K)
@pytest.mark.parametrize("M", GEMM_M)
def test_gemm3x_passes_match_fp64(M, Kx):
    """Forward (N = 64, bias + ReLU; strided x, no bias, no ReLU), dgrad (N = Kx: BN = 112 with 1..8 column tiles), wgrad
    over 1, 21 and 200 row slabs, and the Gemm3xLinearFn glue around them.  M covers tiles below, at and above the 148 SMs
    and an uneven persistent-grid split; every pass must repeat its bits."""
    from torcheasyrec_b200 import dense_gemm as G

    lib = G._gemm3x_lib()
    assert lib is not None, "libtzk_gemm3x.so missing: build() did not produce it"
    g = torch.Generator(device=DEV).manual_seed(M * 1009 + Kx)
    x, sign, _ = _row_scaled(g, M, Kx)
    dz, _, _ = _row_scaled(g, M, 64, sign=sign)           # same row signs: dz^T x sums terms of one sign per element
    w = _ties(g, (64, Kx)) * torch.where(torch.rand(64, 1, generator=g, device=DEV) < 0.5, -1.0, 1.0) / 32
    b = torch.randn(64, generator=g, device=DEV)
    xbuf = torch.full((M, Kx + 16), float("nan"), device=DEV)   # strided x: NaN beyond column Kx must not be read
    xbuf[:, :Kx] = x
    xs = xbuf[:, :Kx]
    wt = w.t().contiguous()
    xg, wg, bg = x.clone().requires_grad_(), w.clone().requires_grad_(), b.clone().requires_grad_()

    def passes():
        out = {"fwd": G.gemm3x(lib, x, w, b, True), "fwd_strided": G.gemm3x(lib, xs, w, None, False),
               "dgrad": G.gemm3x(lib, dz, wt, None, False)}        # dz [M, 64] @ W [64, Kx] with N = Kx
        for slabs in (1, 21, 200):                                  # 200 > M / 32: empty slabs; short last slabs
            out[slabs] = G.wgrad3x(lib, xs, dz, slabs)
        return out

    got, names = _kernels_run(passes)
    for k in ("gemm3x_kernel<64", "gemm3x_kernel<112", "wgrad3x_kernel"):
        assert k in names, names
    again = passes()
    for k, v in got.items():
        assert torch.equal(v, again[k]), f"{k}: bits differ run to run"

    x64, dz64, w64, b64 = x.double(), dz.double(), w.double(), b.double()
    ref = x64 @ w64.T
    ab = x64.abs() @ w64.abs().T
    # |relu(p) - relu(q)| <= |p - q|: the bound of the pre-activation holds after the ReLU
    _check("forward", got["fwd"], torch.relu(ref + b64), _gemm3x_c(Kx) * U * (ab + b64.abs()))
    _check("forward, strided x, no bias, no ReLU", got["fwd_strided"], ref, _gemm3x_c(Kx) * U * ab)
    _check("dgrad", got["dgrad"], dz64 @ w64, _gemm3x_c(64) * U * (dz64.abs() @ w64.abs()))
    ref_w, ab_w = dz64.T @ x64, dz64.abs().T @ x64.abs()
    for slabs in (1, 21, 200):
        _check(f"wgrad, {slabs} slabs", got[slabs], ref_w, _wgrad3x_c(M, slabs) * U * ab_w)

    # the autograd glue: forward + act_bwd_colsum + dgrad + wgrad (SLABS) with the ReLU mask of the fp32 forward
    yg = G.Gemm3xLinearFn.apply(lib, xg, wg, bg, True, None)
    yg.backward(dz)
    assert torch.equal(yg.detach(), got["fwd"])
    dzm = dz64 * (yg.detach() > 0)
    _check("Gemm3xLinearFn dx", xg.grad, dzm @ w64, _gemm3x_c(64) * U * (dzm.abs() @ w64.abs()))
    _check("Gemm3xLinearFn dW", wg.grad, dzm.T @ x64, _wgrad3x_c(M, G.SLABS) * U * (dzm.abs().T @ x64.abs()))
    _check("Gemm3xLinearFn db", bg.grad, dzm.sum(0), _rows_c(M) * U * dzm.abs().sum(0))


# ==========================================================================================================================
# 3. DLRM interaction on the tensor cores (csrc/tzk_interact_tc.cuh) and its FFMA twin (csrc/tzk_dense.cu)
# ==========================================================================================================================
ITC_FWD_C = 3 * 16 + SPLIT + 2   # three MMAs of the split per k-step, K = 16 terms each, into one accumulator
ITC_BWD_C = 3 * 32 + SPLIT + 3   # S X: K = 32 (27 rows padded), three MMAs per k-step; + the pass-through add


def _interaction_inputs(g, B):
    """27 rows of 16 per sample with magnitudes 2^-10 .. 2^10 inside a row and random signs; rows 1..13 are
    antisymmetric in their two halves and row 0 symmetric, so z_0j (j = 1..13) cancels to 0."""
    mag = torch.exp2(torch.randint(-10, 11, (B, 27, 16), generator=g, device=g.device).float())
    sgn = torch.where(torch.rand(B, 27, 16, generator=g, device=g.device) < 0.5, -1.0, 1.0)
    X = _ties(g, (B, 27, 16), generic=0.5) * mag * sgn
    X[:, 0, 8:] = X[:, 0, :8]
    X[:, 1:14, 8:] = -X[:, 1:14, :8]
    return X


@pytest.mark.parametrize("path", ["tc", "ffma"])
@pytest.mark.parametrize("B", [1, 31, 65536, 65537])
def test_dlrm_interaction_matches_fp64(kernels, monkeypatch, B, path):
    """[351 pairs | 0 | 16 dense | 416 sparse] rows: pairs within 3xTF32 / FFMA error of float64 even where they cancel,
    the zero and the copies bit-exact; the backward ignores the pad column's gradient (NaN there)."""
    for v in ("TZK_INTERACT_TC_FWD", "TZK_INTERACT_TC_BWD"):
        monkeypatch.delenv(v, raising=False)
    monkeypatch.setenv("TZK_INTERACT_TC", "1" if path == "tc" else "0")
    g = torch.Generator(device=DEV).manual_seed(B)
    X = _interaction_inputs(g, B)
    d_out = torch.randn(B, 784, generator=g, device=DEV) * \
        torch.exp2(torch.randint(-6, 7, (B, 784), generator=g, device=DEV).float())
    d_out[:, 351] = float("nan")
    dense, sparse = X[:, 0].contiguous(), X[:, 1:].reshape(B, 416).contiguous()

    def fwd():
        return kernels.dot_interact_fwd(dense, sparse, 26, 16, True, True, pad_to=4, p_pad=1)

    def bwd():
        return kernels.dot_interact_bwd(dense, sparse, d_out, 26, 16, True, True, p_pad=1)

    (out, (dd, ds)), names = _kernels_run(lambda: (fwd(), bwd()))
    for k in ("dot_interact27_fwd_tc_kernel", "dot_interact27_bwd_tc_kernel"):
        assert (k in names) == (path == "tc"), names
    for k in ("dot_interact_fwd_kernel", "dot_interact_bwd_kernel"):
        assert (k in names) == (path == "ffma"), names
    assert out.shape == (B, 784)
    assert bool((out[:, 351] == 0).all())
    assert torch.equal(out[:, 352:368], dense) and torch.equal(out[:, 368:], sparse)
    X64 = X.double()
    iu = torch.triu_indices(27, 27, 1, device=DEV)
    z = (X64 @ X64.transpose(1, 2))[:, iu[0], iu[1]]
    ab = (X64.abs() @ X64.abs().transpose(1, 2))[:, iu[0], iu[1]]
    _check("pairs", out[:, :351], z, ITC_FWD_C * U * ab)

    S = torch.zeros(B, 27, 27, dtype=torch.float64, device=DEV)
    S[:, iu[0], iu[1]] = d_out[:, :351].double()
    S = S + S.transpose(1, 2)
    pas = d_out[:, 352:].double().reshape(B, 27, 16)
    dX = S @ X64 + pas
    abX = S.abs() @ X64.abs() + pas.abs()
    _check("d_dense", dd, dX[:, 0], ITC_BWD_C * U * abX[:, 0])
    _check("d_sparse", ds, dX[:, 1:].reshape(B, 416), ITC_BWD_C * U * abX[:, 1:].reshape(B, 416))
    assert torch.equal(fwd(), out)
    dd2, ds2 = bwd()
    assert torch.equal(dd2, dd) and torch.equal(ds2, ds)


# ==========================================================================================================================
# 4. Narrow layers (csrc/tzk_tower.cu, tzk_tower_bwd2.cuh) and the fused tail + BCE (csrc/tzk_tower_tail.cuh)
# ==========================================================================================================================
NARROW_M = [31, 32, 33, 127, 128, 129, 65536]
NARROW_KN = [(1, 1), (1, 64), (64, 1), (64, 64)]


@pytest.mark.parametrize("K,N", NARROW_KN)
@pytest.mark.parametrize("M", NARROW_M)
def test_small_linear_matches_fp64(kernels, monkeypatch, M, K, N):
    """relu(x W^T + b) forward (a row per thread, FFMA in k order: c = K + 1) and dx (c = N), dW, db (row sums) backward;
    bias-free and ReLU-free when N = 1."""
    for v in ("TZK_SMALL_LINEAR_BWD", "TZK_SMALL_LINEAR_DW"):
        monkeypatch.delenv(v, raising=False)
    g = torch.Generator(device=DEV).manual_seed(M * 131 + K * 7 + N)
    relu, has_bias = N != 1, N != 1
    x = _row_scaled(g, M, K)[0]
    w = torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)
    b = torch.randn(N, generator=g, device=DEV) if has_bias else None
    dy = torch.randn(M, N, generator=g, device=DEV)

    def layer():
        y = kernels.small_linear_fwd(x, w, b, relu)
        return (y,) + kernels.small_linear_bwd(x, w, y if relu else None, dy, relu, True, has_bias)

    (y, dx, dw, db), names = _kernels_run(layer)
    for k in ("small_linear_fwd_rows_kernel", "small_linear_dx_rows_kernel", "small_linear_dw_tiles_kernel"):
        assert k in names, names
    x64, w64, dy64 = x.double(), w.double(), dy.double()
    b64 = b.double() if has_bias else torch.zeros(N, dtype=torch.float64, device=DEV)
    ref = x64 @ w64.T + b64
    _check("forward", y, torch.relu(ref) if relu else ref, (K + 1) * U * (x64.abs() @ w64.abs().T + b64.abs()))
    dz = dy64 * (y > 0) if relu else dy64                 # the fp32 forward's own mask: no ReLU tie can flip
    _check("dx", dx, dz @ w64, N * U * (dz.abs() @ w64.abs()))
    _check("dW", dw, dz.T @ x64, _rows_c(M) * U * (dz.abs().T @ x64.abs()))
    if has_bias:
        _check("db", db, dz.sum(0), _rows_c(M) * U * dz.abs().sum(0))
    else:
        assert db is None
    again = layer()
    assert all(torch.equal(a, b_) for a, b_ in zip(again, (y, dx, dw, db)) if a is not None)


def _bce_ref(z, ez, t, M, rows_c):
    """mean BCE-with-logits and dloss/dz = (sigmoid(z) - t) / M with bounds.  A row's term and its gradient take a few
    roundings of their own (exp, log1p, the division, the subtraction, 1/M: 8 U relative to the terms) besides what
    z's error makes of them (|dl/dz| = |sigmoid - t| <= 1, |d2l/dz2| <= 1/4); the mean is a row sum."""
    sig = torch.sigmoid(z)
    terms = z.clamp_min(0) - z * t + torch.log1p(torch.exp(-z.abs()))
    e_terms = (sig - t).abs() * ez + 8 * U * (z.clamp_min(0) + (z * t).abs() + torch.log1p(torch.exp(-z.abs())))
    loss = terms.mean()
    e_loss = e_terms.mean() + (rows_c + 1) * U * terms.abs().mean()
    dz = (sig - t) / M
    e_dz = ez / (4 * M) + 8 * U * (sig + t.abs()) / M
    return loss, e_loss, dz, e_dz


@pytest.mark.parametrize("K,N", [(1, 1), (1, 64), (64, 1), (64, 64), (64, 32)])
@pytest.mark.parametrize("M", NARROW_M)
def test_tower_tail_bce_matches_fp64(kernels, M, K, N):
    """loss, logits and the five gradients of the fused tail.  Soft labels (0.3, 0.7) next to 0 / 1, logits up to
    |z| = 100, b1 / b2 = None in some cases.  y1, W1 and b1 are multiples of 2^-7 small enough for y1 W1^T + b1 to be
    exact in fp32, and b1 an odd multiple of 2^-7 where present: the hidden ReLU's mask is exact (no tie can flip it)."""
    from torcheasyrec_b200 import dense_gemm as G

    g = torch.Generator().manual_seed(M * 17 + K * 3 + N)
    y1 = torch.randint(0, 8, (M, K), generator=g).float() / 8
    w1 = torch.randint(-7, 8, (N, K), generator=g).float() / 8
    has_b1, has_b2 = (K + N) % 2 == 0, N != 64
    b1 = (2 * torch.randint(-16, 16, (N,), generator=g).float() + 1) / 128 if has_b1 else None
    h = torch.relu(y1.double() @ w1.double().T + (b1.double() if has_b1 else 0))
    w2 = torch.randn(1, N, generator=g, dtype=torch.float64)
    w2 = (w2 * 100 / max(float((h @ w2.T).abs().max()), 1e-3)).float()   # logits up to |z| ~ 100
    b2 = torch.tensor([0.25]) if has_b2 else None
    lab = torch.tensor([0.0, 1.0, 0.3, 0.7])[torch.randint(0, 4, (M,), generator=g)]
    y1, w1, w2, lab = y1.to(DEV), w1.to(DEV), w2.to(DEV), lab.to(DEV)
    b1 = b1.to(DEV) if has_b1 else None
    b2 = b2.to(DEV) if has_b2 else None
    assert G.tower_tail_usable(y1, w1, w2, lab)
    outs, names = _kernels_run(lambda: kernels.tower_tail_bce(y1, w1, b1, w2, b2, lab))
    assert "tower_tail_bce_kernel" in names, names
    loss, logits, dy1, dW1, db1, dw2, db2 = outs

    y64, w164, w264, t = y1.double(), w1.double(), w2.double(), lab.double()
    zh = y64 @ w164.T + (b1.double() if has_b1 else 0)
    mask = zh > 0                                          # exact: the pre-activations are exact in fp32
    h = zh * mask
    b264 = b2.double() if has_b2 else torch.zeros(1, dtype=torch.float64, device=DEV)
    z, ez = _mm(h, torch.zeros_like(h), w264.T, torch.zeros_like(w264.T), N + 1, b264, torch.zeros_like(b264))
    z, ez = z[:, 0], ez[:, 0]
    _check("logits", logits, z, ez)
    rc = _rows_c(M)
    l_ref, e_l, dz, e_dz = _bce_ref(z, ez, t, M, rc)
    _check("loss", loss, l_ref, e_l)
    dh = dz[:, None] * w264 * mask                         # one rounding: dz * w2
    e_dh = (e_dz[:, None] * w264.abs() + U * dh.abs()) * mask
    zK, zN = torch.zeros(N, K, dtype=torch.float64, device=DEV), torch.zeros(M, N, dtype=torch.float64, device=DEV)
    ref, e = _mm(dh, e_dh, w164, zK, N)
    _check("dy1", dy1, ref, e)
    ref, e = _mm(dh.T, e_dh.T, y64, torch.zeros_like(y64), rc)
    _check("dW1", dW1, ref, e)
    _check("db1", db1, dh.sum(0), e_dh.sum(0) + rc * U * dh.abs().sum(0))
    ref, e = _mm(dz[None, :], e_dz[None, :], h, zN, rc + 1)   # + the rounding of dz * h
    _check("dw2", dw2, ref, e)
    _check("db2", db2, dz.sum(0, keepdim=True), e_dz.sum(0, keepdim=True) + rc * U * dz.abs().sum(0, keepdim=True))
    again = kernels.tower_tail_bce(y1, w1, b1, w2, b2, lab)
    assert all(torch.equal(a, b_) for a, b_ in zip(again, outs))


# ==========================================================================================================================
# 1. The whole DLRM-Criteo dense step in float64
# ==========================================================================================================================
SWITCHES = ["TZK_FUSED_TAIL", "TZK_INTERACT_TC", "TZK_GEMM3X", "TZK_SMALL_LINEAR"]


def _spy(monkeypatch, calls, obj, name, key, keep=None):
    orig = getattr(obj, name)

    def wrapper(*a, **k):
        calls[key] += 1
        out = orig(*a, **k)
        if keep is not None:
            keep[key] = out
        return out

    monkeypatch.setattr(obj, name, wrapper)


@pytest.mark.parametrize("off", [None] + SWITCHES)
@pytest.mark.parametrize("B", [65536, 257, 384])
def test_dlrm_dense_step_matches_fp64(kernels, monkeypatch, B, off):
    """One train_wrapper + backward of DLRM-Criteo (13 -> 64 -> 16 bottom MLP, 27 x 16 interaction, 783 -> 64 -> 32 final
    MLP, Linear(32, 1), mean BCE) against the model restated in float64 from model.state_dict() and the step's own fp32
    inputs (dense features, pooled embeddings): loss, logits, every dense parameter's gradient, and the gradients into
    the pooled embeddings [B, 416] and into the bottom MLP's output [B, 16].  With every switch on, and with each of
    them off in turn.  ReLU masks are the fp32 step's own; the fused tail's hidden mask is read off its dy1 where the
    float64 pre-activation lies within its bound of 0."""
    from torcheasyrec_b200 import dense_gemm as G
    from torcheasyrec_b200 import functional as Fn
    from torcheasyrec_b200.engine import Pipeline

    for v in SWITCHES + ["TZK_INTERACT_TC_FWD", "TZK_INTERACT_TC_BWD", "TZK_SMALL_LINEAR_BWD", "TZK_SMALL_LINEAR_DW"]:
        monkeypatch.delenv(v, raising=False)
    if off:
        monkeypatch.setenv(off, "0")
    pipe = Pipeline("dlrm_criteo", device=DEV, max_rows=1000, seed=21, capturable=False)
    model = pipe.model
    assert not torch.backends.cuda.matmul.allow_tf32
    sd = model.state_dict()

    calls, keep, cap = Counter(), {}, {}
    _spy(monkeypatch, calls, G.Gemm3xLinearFn, "apply", "gemm3x")
    _spy(monkeypatch, calls, G._LinearFn, "apply", "cublaslt")
    _spy(monkeypatch, calls, kernels, "tower_tail_bce", "tail", keep)
    _spy(monkeypatch, calls, kernels, "dot_interact_fwd", "itc_fwd")
    _spy(monkeypatch, calls, kernels, "dot_interact_bwd", "itc_bwd")
    _spy(monkeypatch, calls, kernels, "small_linear_fwd", "small_fwd")
    _spy(monkeypatch, calls, kernels, "bce_logits_fwd_bwd", "bce")
    orig_interaction = Fn.dlrm_interaction

    def interaction(dense_feat, sparse, *a, **k):
        dense_feat.retain_grad()
        sparse.retain_grad()
        cap["h1"], cap["S"] = dense_feat, sparse
        return orig_interaction(dense_feat, sparse, *a, **k)

    monkeypatch.setattr(Fn, "dlrm_interaction", interaction)
    hooks = []
    for key, mod in (("bottom0", model.dense_mlp.mlp[0]), ("final0", model.final_mlp.mlp[0]),
                     ("final1", model.final_mlp.mlp[1])):
        hooks.append(mod.register_forward_hook(lambda m, inp, out, key=key: cap.__setitem__(key, (inp[0], out))))
    batch = pipe.synthetic_batch(B, seed=B).to(DEV)

    def step():
        loss, (_, preds, _) = pipe.train_wrapper(batch)
        loss.backward()
        return loss, preds

    (loss, preds), names = _kernels_run(step)
    for hk in hooks:
        hk.remove()

    # ---- which kernels served the step
    fused = off != "TZK_FUSED_TAIL"
    want = {"gemm3x": int(off != "TZK_GEMM3X"), "cublaslt": int(off == "TZK_GEMM3X") + 2 * int(off == "TZK_SMALL_LINEAR"),
            "tail": int(fused), "itc_fwd": 1, "itc_bwd": 1, "bce": int(not fused),
            "small_fwd": 0 if off == "TZK_SMALL_LINEAR" else (2 if fused else 4)}
    assert {k: calls[k] for k in want} == want, dict(calls)
    assert ("gemm3x_kernel" in names) == (off != "TZK_GEMM3X"), names
    assert ("wgrad3x_kernel" in names) == (off != "TZK_GEMM3X"), names
    assert ("tower_tail_bce_kernel" in names) == fused, names
    assert ("dot_interact27_fwd_tc_kernel" in names) == (off != "TZK_INTERACT_TC"), names
    assert ("dot_interact27_bwd_tc_kernel" in names) == (off != "TZK_INTERACT_TC"), names
    assert ("small_linear_fwd_rows_kernel" in names) == (off != "TZK_SMALL_LINEAR" or not fused), names

    # ---- c of each layer on the path that served it
    rc = _rows_c(B)
    small = off != "TZK_SMALL_LINEAR"
    g3 = off != "TZK_GEMM3X"
    # cuBLASLt BF16x9: every fp32 operand is three bf16 pieces, nine exact partial products per term, summed in an
    # order the library does not document: c = 9 x the summation length (+ the bias / colsum kernels' own)
    c_bot_fwd = (lambda K: K + 1) if small else (lambda K: 9 * K + 2)
    c_bot_dx = (lambda N: N) if small else (lambda N: 9 * N)
    c_bot_dw = rc if small else 9 * B
    c_f0_fwd = _gemm3x_c(784) if g3 else 9 * 784 + 2
    c_f0_dx = _gemm3x_c(64) if g3 else 9 * 64
    c_f0_dw = _wgrad3x_c(B, G.SLABS) if g3 else 9 * B

    def Z(*shape):
        return torch.zeros(*shape, dtype=torch.float64, device=DEV)

    def p(name):
        return sd[name].detach().double()

    W0, b0 = p("dense_mlp.mlp.0.perceptron.0.weight"), p("dense_mlp.mlp.0.perceptron.0.bias")
    W1, b1 = p("dense_mlp.mlp.1.perceptron.0.weight"), p("dense_mlp.mlp.1.perceptron.0.bias")
    F0, c0 = p("final_mlp.mlp.0.perceptron.0.weight"), p("final_mlp.mlp.0.perceptron.0.bias")
    F1, c1 = p("final_mlp.mlp.1.perceptron.0.weight"), p("final_mlp.mlp.1.perceptron.0.bias")
    O, o = p("output_mlp.weight"), p("output_mlp.bias")
    xd = cap["bottom0"][0].detach().double()
    S = cap["S"].detach().double()
    t = batch.labels[model._label_name].double()
    m0 = cap["bottom0"][1].detach() > 0
    m1 = cap["h1"].detach() > 0
    mq0 = cap["final0"][1].detach() > 0

    # ---- forward
    a0, e = _mm(xd, Z(B, 13), W0.T, Z(13, 64), c_bot_fwd(13), b0, Z(64))
    h0, e_h0 = a0 * m0, e * m0
    a1, e = _mm(h0, e_h0, W1.T, Z(64, 16), c_bot_fwd(64), b1, Z(16))
    h1, e_h1 = a1 * m1, e * m1
    X = torch.cat([h1[:, None], S.reshape(B, 26, 16)], 1)
    eX = torch.cat([e_h1[:, None], Z(B, 26, 16)], 1)
    iu = torch.triu_indices(27, 27, 1, device=DEV)
    P, eP = _mm(X, eX, X.transpose(1, 2), eX.transpose(1, 2), ITC_FWD_C)
    f = torch.cat([P[:, iu[0], iu[1]], h1, S], 1)                      # the reference's 783 columns, no zero column
    ef = torch.cat([eP[:, iu[0], iu[1]], e_h1, Z(B, 416)], 1)
    g0, e = _mm(f, ef, F0.T, Z(783, 64), c_f0_fwd, c0, Z(64))
    q0, e_q0 = g0 * mq0, e * mq0
    g1, e_g1 = _mm(q0, e_q0, F1.T, Z(64, 32), 64 + 1, c1, Z(32))      # FFMA in k order from the bias (both paths)
    if fused:
        mq1 = g1 > 0
        dy1 = keep["tail"][2].double()
        amb = g1.abs() <= e_g1
        sig_dz = (torch.sigmoid(g1.clamp_min(0) @ O.T + o)[:, 0] - t) / B      # only to rank the candidates
        one = amb.sum(1) == 1                    # rows with one such pre-activation: both candidates at once
        if bool(one.any()):
            r = one.nonzero().flatten()
            n = amb[r].int().argmax(1)
            base = (sig_dz[r, None] * O[0] * mq1[r] * ~amb[r]) @ F1
            with_n = base + (sig_dz[r] * O[0, n])[:, None] * F1[n]
            take = (with_n - dy1[r]).abs().amax(1) < (base - dy1[r]).abs().amax(1)
            mq1[r, n] = take
        for r in (amb.sum(1) > 1).nonzero().flatten().tolist():
            cols = amb[r].nonzero().flatten().tolist()
            assert len(cols) <= 8, f"row {r}: {len(cols)} hidden pre-activations within their bound of 0"
            best = None
            for bits in itertools.product([False, True], repeat=len(cols)):
                m = mq1[r].clone()
                m[cols] = torch.tensor(bits, device=DEV)
                d = float(((sig_dz[r] * O[0] * m) @ F1 - dy1[r]).abs().max())
                if best is None or d < best[0]:
                    best = (d, m)
            mq1[r] = best[1]
    else:
        mq1 = cap["final1"][1].detach() > 0
    q1, e_q1 = g1 * mq1, e_g1 * mq1
    z, ez = _mm(q1, e_q1, O.T, Z(32, 1), 32 + 1, o, Z(1))
    z, ez = z[:, 0], ez[:, 0]
    _check("logits", preds["logits"], z, ez)
    l_ref, e_l, dz, e_dz = _bce_ref(z, ez, t, B, rc)
    _check("loss", loss, l_ref, e_l)

    # ---- backward
    grads = {}
    grads["output_mlp.weight"] = _mm(dz[None, :], e_dz[None, :], q1, e_q1, rc + 1)
    grads["output_mlp.bias"] = (dz.sum(0, keepdim=True), e_dz.sum(0, keepdim=True) + rc * U * dz.abs().sum(0, keepdim=True))
    dg1 = dz[:, None] * O * mq1
    e_dg1 = (e_dz[:, None] * O.abs() + U * dg1.abs()) * mq1
    grads["final_mlp.mlp.1.perceptron.0.weight"] = _mm(dg1.T, e_dg1.T, q0, e_q0, rc)
    grads["final_mlp.mlp.1.perceptron.0.bias"] = (dg1.sum(0), e_dg1.sum(0) + rc * U * dg1.abs().sum(0))
    dq0, e = _mm(dg1, e_dg1, F1, Z(32, 64), 32)
    dg0, e_dg0 = dq0 * mq0, e * mq0
    grads["final_mlp.mlp.0.perceptron.0.weight"] = _mm(dg0.T, e_dg0.T, f, ef, c_f0_dw)
    grads["final_mlp.mlp.0.perceptron.0.bias"] = (dg0.sum(0), e_dg0.sum(0) + rc * U * dg0.abs().sum(0))
    df, e_df = _mm(dg0, e_dg0, F0, Z(64, 783), c_f0_dx)
    Sm, eSm = Z(B, 27, 27), Z(B, 27, 27)
    Sm[:, iu[0], iu[1]], eSm[:, iu[0], iu[1]] = df[:, :351], e_df[:, :351]
    Sm, eSm = Sm + Sm.transpose(1, 2), eSm + eSm.transpose(1, 2)
    dX, e_dX = _mm(Sm, eSm, X, eX, ITC_BWD_C, df[:, 351:].reshape(B, 27, 16), e_df[:, 351:].reshape(B, 27, 16))
    _check("d pooled embeddings [B, 416]", cap["S"].grad, dX[:, 1:].reshape(B, 416), e_dX[:, 1:].reshape(B, 416))
    _check("d bottom MLP output [B, 16]", cap["h1"].grad, dX[:, 0], e_dX[:, 0])
    da1, e_da1 = dX[:, 0] * m1, e_dX[:, 0] * m1
    grads["dense_mlp.mlp.1.perceptron.0.weight"] = _mm(da1.T, e_da1.T, h0, e_h0, c_bot_dw)
    grads["dense_mlp.mlp.1.perceptron.0.bias"] = (da1.sum(0), e_da1.sum(0) + rc * U * da1.abs().sum(0))
    dh0, e = _mm(da1, e_da1, W1, Z(16, 64), c_bot_dx(16))
    da0, e_da0 = dh0 * m0, e * m0
    grads["dense_mlp.mlp.0.perceptron.0.weight"] = _mm(da0.T, e_da0.T, xd, Z(B, 13), c_bot_dw)
    grads["dense_mlp.mlp.0.perceptron.0.bias"] = (da0.sum(0), e_da0.sum(0) + rc * U * da0.abs().sum(0))

    named = dict(model.named_parameters())
    dense_names = {n for n, q in named.items() if any(q is d for d in model.dense_parameters())}
    assert dense_names == set(grads), sorted(dense_names ^ set(grads))
    for n, (ref, bound) in grads.items():
        assert named[n].grad is not None, n
        _check(n, named[n].grad, ref, bound)
