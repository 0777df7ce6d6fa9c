"""The fused corpus-side encoder's kernels (dkd_mha_small, dkd_linear_exact = dkd_exact_umma.cu mode 4,
dkd_layernorm_rows, dkd_row_stats) and encoder.FusedContextEncoder end to end, over their whole shape range, against
float64 references written here.

Tolerances are derived from each kernel's fp32 error model, per output, from the inputs (U = 2^-24 is the unit roundoff
of fp32): a kernel that is subtly wrong (a scale off by 1e-3, a K block or a bias column off by one, a stale row
statistic) lands far outside them, and each bound's derivation sits next to it.  Shapes that depend on the number of SMs
(the work-item schedule of dkd_linear_exact) are derived from the device so that every regime named here is hit."""
import copy
import math

import pytest
import torch

from oracle import ref_shim

pytestmark = pytest.mark.gpu

U = 2.0 ** -24            # fp32 unit roundoff: |fl(x) - x| <= U |x|
ULP1 = 2.0 ** -23         # ulp(x) <= ULP1 |x|
GRID = 2.0 ** -10         # fp32 spacing in [8192, 16384): where every masked logit s - 10000 lies
TOL = 1e-4                # stated tolerance of the fused encoder on O(1) features (tests/test_gpu_encoder.py)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _call_raw(name, *args):
    from dkd_b200 import _lib
    _lib.call(name, *args)


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ============================================================================================== 1. mha_small
MHA_CASES = [(dh, L, heads) for dh in (16, 32, 64, 96, 128) for L in (1, 2, 31, 32, 33, 77, 127, 128)
             for heads in ((1, 4, 8) if dh <= 64 else (1, 4))]


def _heads_of(qkv, Nv, L, heads, dh, off):
    """(Nv * L, ld) columns [off, off + heads * dh) -> (Nv, heads, L, dh) float64."""
    return qkv[:, off:off + heads * dh].double().reshape(Nv, L, heads, dh).transpose(1, 2)


def _to_rows(t):
    """(Nv, heads, L, dh) -> (Nv * L, heads * dh)."""
    Nv, heads, L, dh = t.shape
    return t.transpose(1, 2).reshape(Nv * L, heads * dh)


def _mha_reference(qkv, Nv, L, heads, dh, keep, q_off, k_off, v_off):
    """float64 softmax(q k^T / sqrt(dh) + (1 - mask) * -10000) v and the kernel's error bound, both (Nv * L, heads * dh);
    plus the rows of fully masked videos, their reference and bound (see below)."""
    q, k, v = (_heads_of(qkv, Nv, L, heads, dh, o) for o in (q_off, k_off, v_off))
    dev = qkv.device
    keep = torch.ones(Nv, L, dtype=torch.bool, device=dev) if keep is None else keep
    kk = keep[:, None, None, :]                                     # (Nv, 1, 1, L) key is valid
    scale = 1.0 / math.sqrt(dh)
    s = q @ k.transpose(-1, -2) * scale
    s_abs = q.abs() @ k.abs().transpose(-1, -2) * scale
    logits = s + (~kk) * -10000.0
    p = torch.softmax(logits, -1)
    ref = p @ v
    # Rows with a valid key.  The kernel's fp32 logit is off by at most
    #   delta_l = dh U sum_d |q_d k_d| scale   (fp32 dot product, gamma_dh)  + 2 U |s_l|  (the scale product, fp32 scale)
    # so exp(a_l - max) is good to the relative rho_l = delta_l + delta_max + __expf's documented (2 + 1.16 |x|) ulp
    # + U |x| (the subtraction), x = a_l - max.  Masked keys of such a row sit ~10000 below the maximum: their weights
    # are exactly 0 in fp32 and float64 alike.  The normalised weights are good to rho_l + max rho + (L + 2) U (sum,
    # reciprocal, product) and the fmaf weighted sum adds L U sum_l p_l |v_l|, so
    #   |out - ref| <= (2 max_l rho_l + (2 L + 2) U) * sum_l p_l |v_l|.
    delta = (dh * U * s_abs + 2 * U * s.abs()).masked_fill(~kk, 0.0)
    x = (logits - logits.amax(-1, keepdim=True)).abs()
    rho = (delta + (2 + 1.16 * x) * ULP1 + U * x).masked_fill(~kk, 0.0).amax(-1, keepdim=True) + delta.amax(-1, keepdim=True)
    pv = p @ v.abs()
    tol = (2 * rho + (2 * L + 2) * U) * pv
    # Fully masked videos.  Every logit is s - 10000, where the fp32 grid is GRID = 2^-10: any fp32 implementation
    # (the PyTorch mirror included) gets the weights only to ~1e-3 relative.  Reference: float64 softmax of the
    # fp32-rounded logits fl(fl(s) - 10000).  The kernel's score differs from s by delta << GRID, so its rounded logit is
    # the reference's or the grid point next to it: each logit moves by at most GRID, each weight (a logit over a sum of
    # them) by at most a factor exp(2 GRID), and the output by expm1(2 GRID) sum_l p_l |v_l|; the differences a_l - max
    # are exact (multiples of GRID), so the fp32 part is the valid-row bound with delta = 0.
    dead = ~keep.any(1)                                             # (Nv,) fully masked videos
    a32 = (s.float().double() - 10000.0).float().double()
    p32 = torch.softmax(a32, -1)
    ref_dead = p32 @ v
    pv32 = p32 @ v.abs()
    x32 = (a32 - a32.amax(-1, keepdim=True)).abs()
    rho32 = ((2 + 1.16 * x32) * ULP1 + U * x32).amax(-1, keepdim=True)
    tol_dead = (math.expm1(2 * GRID) + 2 * rho32 + (2 * L + 2) * U) * pv32
    return _to_rows(ref), _to_rows(tol), dead, _to_rows(ref_dead), _to_rows(tol_dead)


def _mha_mirror_fp32(qkv, Nv, L, heads, dh, keep):
    """The model's fp32 PyTorch attention (model._SelfAttention.forward) on the default layout."""
    H = heads * dh
    split = lambda t: t.reshape(Nv, L, heads, dh).transpose(1, 2)  # noqa: E731
    q, k, v = split(qkv[:, :H]), split(qkv[:, H:2 * H]), split(qkv[:, 2 * H:3 * H])
    att = q @ k.transpose(-1, -2) / math.sqrt(dh)
    att = att + (1 - keep.float()[:, None, None, :]) * -10000.0
    return _to_rows(torch.softmax(att, dim=-1) @ v)


def _check_mha(got, Nv, L, ref, tol, dead, ref_dead, tol_dead, what):
    rows_dead = dead.repeat_interleave(L)
    live = ~rows_dead
    err = (got.double() - ref).abs()
    assert bool((err[live] <= tol[live]).all()), (
        f"{what}: valid rows off by {float(err[live].max()):.3g}, worst / bound {float((err / tol)[live].max()):.3g}")
    if bool(rows_dead.any()):
        err_d = (got.double() - ref_dead).abs()[rows_dead]
        assert bool((err_d <= tol_dead[rows_dead]).all()), (
            f"{what}: fully masked rows off by {float(err_d.max()):.3g} (bound {float(tol_dead[rows_dead].max()):.3g})")


def _mha_inputs(Nv, L, heads, dh, seed, ld=None):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ld = 3 * heads * dh if ld is None else ld
    qkv = torch.randn(Nv * L, ld, device="cuda", generator=g)
    # video 0: every frame; video 1: a random length (1 .. L); video 2: one frame; video 3: no frame at all
    lens = torch.tensor([L, int(torch.randint(1, L + 1, (1,), generator=g, device="cuda")), 1, 0], device="cuda")[:Nv]
    keep = torch.arange(L, device="cuda")[None] < lens[:, None]
    return qkv, keep


@pytest.mark.parametrize("dh,L,heads", MHA_CASES)
def test_mha_small_against_float64(ops, dh, L, heads):
    Nv, H = 4, heads * dh
    qkv, keep = _mha_inputs(Nv, L, heads, dh, seed=1000 * dh + 10 * L + heads)
    for mask in (None, keep):
        m8 = None if mask is None else mask.to(torch.uint8).contiguous()
        got = ops.mha_small(qkv, Nv, L, heads, dh, m8)
        ref, tol, dead, ref_d, tol_d = _mha_reference(qkv, Nv, L, heads, dh, mask, 0, H, 2 * H)
        _check_mha(got, Nv, L, ref, tol, dead, ref_d, tol_d, f"dh={dh} L={L} heads={heads} mask={mask is not None}")
        if mask is not None:
            # the fully masked video is ill-conditioned in any fp32 implementation: the kernel sits within the same
            # one-grid-step bound of the fp32 PyTorch mirror as of the float64 reference
            rows_dead = dead.repeat_interleave(L)
            mirror = _mha_mirror_fp32(qkv, Nv, L, heads, dh, mask)
            assert bool(((got - mirror).abs().double()[rows_dead] <= tol_d[rows_dead]).all())


@pytest.mark.parametrize("dh", (16, 32, 64, 96, 128))
def test_mha_small_custom_layout_leaves_other_columns(ops, dh):
    """q / k / v at offsets of a wider row (v first), output into a wider buffer through the C ABI: the columns past
    heads * dh keep their sentinels."""
    Nv, L, heads = 4, 77, 4
    H = heads * dh
    v_off, q_off, k_off = 4, H + 12, 2 * H + 20
    ld = k_off + H                                  # the last block ends exactly at the row's end
    qkv, keep = _mha_inputs(Nv, L, heads, dh, seed=dh, ld=ld)
    m8 = keep.to(torch.uint8).contiguous()
    out_ld = H + 12
    sentinel = -12345.5
    out = torch.full((Nv * L, out_ld), sentinel, device="cuda")
    _call_raw("dkd_mha_small", qkv.data_ptr(), ld, q_off, k_off, v_off, m8.data_ptr(), Nv, L, heads, dh,
              1.0 / float(dh) ** 0.5, out.data_ptr(), out_ld, _stream())
    assert bool((out[:, H:] == sentinel).all())
    ref, tol, dead, ref_d, tol_d = _mha_reference(qkv, Nv, L, heads, dh, keep, q_off, k_off, v_off)
    _check_mha(out[:, :H], Nv, L, ref, tol, dead, ref_d, tol_d, f"custom layout dh={dh}")


def test_mha_small_rejects_inconsistent_layout(ops):
    """DKD_ERR_SHAPE for a negative offset, a q / k / v block past the row's end, an output row narrower than
    heads * dh.  The buffers are padded so that even an unchecked launch of every case would stay inside them; the
    output keeps its sentinel (nothing ran)."""
    from dkd_b200 import _lib
    Nv, L, heads, dh = 2, 16, 4, 32
    H = heads * dh
    pad = 4 * H                                     # floats of slack on both sides of every buffer
    qkv_buf = torch.zeros(Nv * L * 3 * H + 2 * pad, device="cuda")
    out_buf = torch.full((Nv * L * H + 2 * pad,), 7.0, device="cuda")
    qkv_p, out_p = qkv_buf.data_ptr() + 4 * pad, out_buf.data_ptr() + 4 * pad
    bad = [
        (3 * H, -4, H, 2 * H, H),                   # q_off < 0
        (3 * H, 0, -4, 2 * H, H),                   # k_off < 0
        (3 * H, 0, H, -4, H),                       # v_off < 0
        (3 * H - 4, 0, H, 2 * H, H),                # v block runs 4 columns past ld
        (3 * H, 4, H, 2 * H + 4, H),                # v block runs 4 columns past ld (offsets shifted)
        (3 * H, 0, H, 2 * H, H - 4),                # out_ld < heads * dh
    ]
    for ld, qo, ko, vo, out_ld in bad:
        with pytest.raises(_lib.DkdError, match="code -2"):
            _call_raw("dkd_mha_small", qkv_p, ld, qo, ko, vo, None, Nv, L, heads, dh, 0.125, out_p, out_ld, _stream())
    torch.cuda.synchronize()
    assert bool((out_buf == 7.0).all())


# ============================================================================================== 2. linear_exact
def _schedule(M, N, sms):
    """dkd_linear_exact's work items: (tiles_per_chunk, chunks, items, tiles of the last chunk)."""
    wtiles, tiles = -(-N // 128), -(-M // 128)
    chunks = min(tiles, max(1, -(-6 * sms // wtiles)))            # the C loop: ++chunks while < tiles and < 6 SMs
    tpc = -(-tiles // chunks)
    tile_chunks = -(-tiles // tpc)
    return tpc, tile_chunks, wtiles * tile_chunks, tiles - (tile_chunks - 1) * tpc


def _xhat(x, ss):
    xh = x.double()
    return xh if ss is None else xh * ss[:, :1].double() + ss[:, 1:].double()


def _linear_reference(x, w, bias, relu, ss):
    """float64 act(x_hat W^T + b) and the per-output bound of the tf32 x 3 tensor-core GEMM.

    Every product is split into hi.hi + hi.lo + lo.hi (3 tcgen05.mma per 8 features, small terms first), each good to
    2^-21 relative, and the fp32 TMEM accumulator truncates: each MMA loses at most one ulp of the running sum.  Between
    the 8-feature boundaries b-1 and b the running sum is at most max(|P(b-1)|, |P(b)|) + sum over the block of
    |x_hat_k w_k|, P(b) the float64 prefix sum, so
      tol = 3 ulp1 (sum_b max(|P(b-1)|, |P(b)|) + sum_k |x_hat_k w_k|) + 2^-20 sum_k |x_hat_k w_k| + ulp(out)
    (the 2^-20 term also covers the stager's x * scale + shift fma, 2^-24 relative, and the bias addition is in the
    last ulp).  P is built as K / 8 rank-8 updates in float64."""
    xh, wd = _xhat(x, ss), w.double()
    M, K = xh.shape
    S = torch.zeros(M, w.shape[0], dtype=torch.float64, device=x.device)
    prev, walk = torch.zeros_like(S), torch.zeros_like(S)
    for b0 in range(0, K, 8):
        S.addmm_(xh[:, b0:b0 + 8], wd[:, b0:b0 + 8].T)
        a = S.abs()
        walk += torch.maximum(a, prev)
        prev = a
    absprod = xh.abs() @ wd.abs().T
    pre = S if bias is None else S + bias.double()
    tol = 3 * ULP1 * (walk + absprod) + 2.0 ** -20 * absprod + ULP1 * pre.abs()
    return (pre.clamp_min(0) if relu else pre), tol, xh


def _assert_bound_is_sharp(tol, xh, w, bias):
    """The bound must catch the mistakes it exists for: dropping the last K block or reading the bias one column off
    changes almost every output by more than the bound."""
    K = xh.shape[1]
    drop = (xh[:, K - 32:] @ w.double()[:, K - 32:].T).abs()
    assert float((drop > 4 * tol).double().mean()) > 0.9
    if bias is not None and bias.numel() > 1:
        shift = (bias.double() - bias.double().roll(1)).abs()[None]
        assert float((shift > 4 * tol).double().mean()) > 0.9


LIN_VARIANTS = [(False, False, False), (True, False, True), (False, True, False), (True, True, True)]   # bias, relu, ss


def _linear_inputs(M, K, N, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(M, K, device="cuda", generator=g)
    w = torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)
    bias = torch.randn(N, device="cuda", generator=g)
    # an arbitrary per-row (scale, shift): the prologue is x * scale + shift whatever produced the pair
    ss = torch.stack([0.5 + 1.5 * torch.rand(M, device="cuda", generator=g),
                      torch.randn(M, device="cuda", generator=g)], 1).contiguous()
    return x, w, bias, ss


def _check_linear(ops, x, planes, N, bias, relu, ss, ref, tol, what, extra=8):
    """Run into a wider output buffer (ld_out = N + extra) and check every output and the untouched columns."""
    M = x.shape[0]
    sentinel = -777.25
    out = torch.full((M, N + extra), sentinel, device="cuda")
    ops.linear_exact(x, planes, N, bias=bias, relu=relu, row_scale_shift=ss, out=out)
    assert bool((out[:, N:] == sentinel).all()), f"{what}: columns past N written"
    err = (out[:, :N].double() - ref).abs()
    assert bool((err <= tol).all()), f"{what}: off by {float(err.max()):.3g}, worst / bound {float((err / tol).max()):.3g}"


@pytest.mark.parametrize("N", (4, 36, 128, 132, 384, 768, 1152))
@pytest.mark.parametrize("K", (32, 96, 384, 1024, 3072))
def test_linear_exact_against_float64(ops, K, N):
    Mmax = 1000
    x, w, bias, ss = _linear_inputs(Mmax, K, N, seed=K * 10000 + N)
    planes = ops.pack_weight(w)
    for use_b, relu, use_ss in LIN_VARIANTS:
        b_, s_ = (bias if use_b else None), (ss if use_ss else None)
        ref, tol, xh = _linear_reference(x, w, b_, relu, s_)
        if not relu:
            _assert_bound_is_sharp(tol, xh, w, b_)
        for M in (1, 127, 128, 129, Mmax):
            _check_linear(ops, x[:M], planes, N, b_, relu, None if s_ is None else s_[:M], ref[:M], tol[:M],
                          f"M={M} K={K} N={N} bias={use_b} relu={relu} ss={use_ss}")


def _rows_for(regime, N, sms):
    """Row count that puts dkd_linear_exact in the named regime of its work-item schedule on this device."""
    for tiles in range(1, 40 * sms):
        M = tiles * 128 - 37                                       # ragged last tile as well
        tpc, chunks, items, last = _schedule(M, N, sms)
        if regime == "one_tile_items" and tpc == 1 and items >= 2 * sms + 1:
            return M
        if regime == "multi_tile_ragged" and tpc >= 2 and last < tpc:
            return M
    raise AssertionError(f"no row count gives {regime} for N = {N} on {sms} SMs")


@pytest.mark.parametrize("regime,N", [("one_tile_items", 128), ("multi_tile_ragged", 128), ("multi_tile_ragged", 768)])
def test_linear_exact_multi_tile_schedule(ops, regime, N):
    """Work items of several 128-row tiles with a ragged last chunk (the per-tile row scale / shift cache, the
    (tile, K block) walk of the stagers across tiles with an odd number of K blocks, the A-ring counter across items),
    and items of one tile each with several items per CTA (the cache must be reset between items)."""
    sms, K = _sms(), 96
    M = _rows_for(regime, N, sms)
    tpc, chunks, items, last = _schedule(M, N, sms)
    assert items > sms and (tpc == 1 if regime == "one_tile_items" else (tpc >= 2 and last < tpc))
    x, w, bias, ss = _linear_inputs(M, K, N, seed=M)
    planes = ops.pack_weight(w)
    for use_b, relu, use_ss in ((True, True, True), (False, False, False), (True, False, True)):
        b_, s_ = (bias if use_b else None), (ss if use_ss else None)
        ref, tol, xh = _linear_reference(x, w, b_, relu, s_)
        _check_linear(ops, x, planes, N, b_, relu, s_, ref, tol,
                      f"{regime} M={M} N={N} tpc={tpc} items={items} bias={use_b} relu={relu} ss={use_ss}")


def test_linear_exact_tvr_corpus_schedule(ops):
    """The production call: the TVR corpus (2,179 videos x 128 frames) through the input projection of both branches
    (K = 3072, N = 768) with the LayerNorm prologue, bias and ReLU.  The per-output bound is checked on every row of the
    first and the last chunk and on a random sample; every output meets the looser bound that replaces each prefix sum
    by sum_k |x_hat_k w_k|."""
    sms, M, K, N = _sms(), 2179 * 128, 3072, 768
    tpc, chunks, items, last = _schedule(M, N, sms)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(M, K, device="cuda", generator=g)
    x = x / x.norm(dim=1, keepdim=True)                            # L2-normalised rows, like the real features
    w = 0.02 * torch.randn(N, K, device="cuda", generator=g)
    bias = torch.randn(N, device="cuda", generator=g)
    ss = ops.row_stats(x, 1e-5)
    out = ops.linear_exact(x, ops.pack_weight(w), N, bias=bias, relu=True, row_scale_shift=ss)
    rows_chunk = tpc * 128
    sample = torch.cat([torch.arange(0, rows_chunk, device="cuda"),
                        torch.arange((chunks - 1) * rows_chunk, M, device="cuda"),
                        torch.randint(0, M, (2048,), device="cuda", generator=g)])
    ref, tol, _ = _linear_reference(x[sample], w, bias, True, ss[sample])
    err = (out[sample].double() - ref).abs()
    assert bool((err <= tol).all()), f"tpc={tpc}: off by {float(err.max()):.3g}, worst / bound {float((err / tol).max()):.3g}"
    wd = w.double()
    loose = 3 * ULP1 * (K // 8 + 1) + 2.0 ** -20
    for r0 in range(0, M, 16384):
        xh = _xhat(x[r0:r0 + 16384], ss[r0:r0 + 16384])
        pre = xh @ wd.T + bias.double()
        tol_g = loose * (xh.abs() @ wd.abs().T) + ULP1 * pre.abs()
        assert bool(((out[r0:r0 + 16384].double() - pre.clamp_min(0)).abs() <= tol_g).all()), f"rows {r0}.."


# ============================================================================================== 3. LayerNorm kernels
def _ln_bound(v, S, n_adds, depth, eps):
    """float64 LayerNorm statistics of v (rows, D) and the fp32 error bounds of a kernel that forms v from n_adds fp32
    additions of terms whose absolute values sum to S, then sums each row along a tree of `depth` rounding levels.
    Returns mean, rstd, a = v - mean, E_mean (error of the kernel's mean), E_a (of its a = v - mean), E_rstd (relative
    error of its rstd)."""
    D = v.shape[1]
    mean = v.mean(1, keepdim=True)
    a = v - mean
    var = (a * a).mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    E_v = n_adds * U * S
    E_mean = depth * U * S.mean(1, keepdim=True) + E_v.mean(1, keepdim=True) + U * mean.abs()   # sum (gamma_depth), / D
    E_own = E_v + U * a.abs()                                      # per element: its input sums, the subtraction
    E_a = E_own + E_mean
    # q = sum (a + da)^2 with da = -dmean + e: the row-wide mean error cancels to first order (sum a = 0), leaving
    # 2 |a| E_own + E_a^2; the squares and their tree add (depth + 3) U q; then / D, + eps and rsqrtf (2 ulp):
    # rstd = (q / D + eps)^(-1/2) halves the relative error of its argument
    dq = (2 * a.abs() * E_own + E_a * E_a).mean(1, keepdim=True) + (depth + 3) * U * var
    E_rstd = 0.5 * dq / (var + eps) + U * (var / (var + eps)) + 2 * ULP1
    return mean, rstd, a, E_mean, E_a, E_rstd


@pytest.mark.parametrize("D", (4, 36, 64, 128, 384, 508, 512))
def test_layernorm_rows_against_float64(ops, D):
    g = torch.Generator(device="cuda").manual_seed(D)
    R, L, eps = 1000, 6, 1e-5                                      # L divides none of the row counts below
    xw = torch.randn(R, D + 12, device="cuda", generator=g)
    xw[3, 8:8 + D] = 0.75                                          # a constant row: variance 0, rstd = 1 / sqrt(eps)
    x = xw[:, 8:8 + D]                                             # x_ld = D + 12
    rw = torch.randn(R, D + 4, device="cuda", generator=g)
    res = rw[:, 4:4 + D]                                           # res_ld = D + 4
    pos_table = torch.randn(L + 3, D, device="cuda", generator=g)  # more rows than L: only the first L are read
    gamma = 1.0 + 0.5 * torch.randn(D, device="cuda", generator=g)
    beta = torch.randn(D, device="cuda", generator=g)
    # layernorm_rows sums each lane's (up to 4) float4s ((x + y) + (z + w)), then a 5-level warp tree
    depth = 2 + 4 + 5
    for rows in (1, 7, 8, 9, R):
        idx = torch.arange(rows, device="cuda")
        for use_pos, use_res in ((False, False), (True, False), (False, True), (True, True)):
            got = ops.layernorm_rows(x[:rows], gamma, beta, eps, residual=res[:rows] if use_res else None,
                                     pos=pos_table if use_pos else None, L=L if use_pos else 0)
            v, S = x[:rows].double(), x[:rows].double().abs()
            if use_pos:
                pr = pos_table[:L].double()[idx % L]
                v, S = v + pr, S + pr.abs()
            if use_res:
                v, S = v + res[:rows].double(), S + res[:rows].double().abs()
            mean, rstd, a, _, E_a, E_rstd = _ln_bound(v, S, int(use_pos) + int(use_res), depth, eps)
            y = a * rstd * gamma.double() + beta.double()
            # y = ((v - mean) rstd) gamma + beta: the error of a and of rstd, then three more roundings
            tol = gamma.double().abs() * rstd * (E_a + a.abs() * E_rstd) + 3 * U * (a * rstd * gamma.double()).abs() \
                + U * y.abs()
            err = (got.double() - y).abs()
            what = f"D={D} rows={rows} pos={use_pos} res={use_res}"
            assert bool((err <= tol).all()), f"{what}: off by {float(err.max()):.3g}, worst / bound {float((err / tol).max()):.3g}"
            if rows > 3 and not use_pos and not use_res:
                assert torch.equal(got[3], beta), what                 # constant row: exactly beta


@pytest.mark.parametrize("D", (4, 48, 1024, 3072, 4100))
def test_row_stats_against_float64(ops, D):
    g = torch.Generator(device="cuda").manual_seed(D)
    rows, eps = 77, 1e-5
    x = 0.3 * torch.randn(rows, D, device="cuda", generator=g) + torch.randn(rows, 1, device="cuda", generator=g)
    x[5] = 0.75                                                   # constant row
    got = ops.row_stats(x, eps)
    xd = x.double()
    depth = 2 + -(-(D // 4) // 32) + 5                             # float4 pair sums, the lane's loop, the warp tree
    mean, rstd, a, E_mean, _, E_rstd = _ln_bound(xd, xd.abs(), 0, depth, eps)
    rs, sh = got[:, :1].double(), got[:, 1:].double()
    assert bool(((rs - rstd).abs() <= E_rstd * rstd).all()), f"D={D}: rstd off by {float(((rs - rstd) / rstd).abs().max()):.3g}"
    want_sh = -mean * rstd
    tol_sh = rstd * E_mean + (mean * rstd).abs() * (E_rstd + U)
    assert bool(((sh - want_sh).abs() <= tol_sh).all()), f"D={D}: shift off by {float((sh - want_sh).abs().max()):.3g}"
    assert float(got[5, 0]) == pytest.approx(1 / math.sqrt(eps), rel=4 * ULP1)
    assert float(got[5, 1]) == pytest.approx(-0.75 / math.sqrt(eps), rel=4 * ULP1)


def test_layernorm_prologue_folded_shift_error(ops):
    """The projection's stager applies the LayerNorm as fma(x, rstd, -mean * rstd).  The folded shift is rounded
    (2^-24 |mean| rstd) and the fp32 mean is good to gamma_depth |mean| (the unfolded (x - mean) rstd shares that), so
    the prologue's error grows with |mean| / std:  ~ (depth + 1) 2^-24 |mean| rstd + O(2^-20) |x_hat|.  Real features
    (L2-normalised rows) sit near |mean| / std ~ 1; the rows here go to 10^3, where the bound passes the encoder's
    1e-4.  Up to 10 the error stays far below it."""
    D, eps = 128, 1e-5
    g = torch.Generator(device="cuda").manual_seed(3)
    ratios = torch.tensor([1.0, 10.0, 100.0, 1000.0], device="cuda").repeat_interleave(64)
    sigma = 0.05 * (1 + torch.rand(ratios.numel(), 1, device="cuda", generator=g))
    sign = torch.where(torch.rand(ratios.numel(), 1, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    x = sigma * (sign * ratios[:, None] + torch.randn(ratios.numel(), D, device="cuda", generator=g))
    ss = ops.row_stats(x, eps)
    eye = torch.eye(D, device="cuda")
    got = ops.linear_exact(x, ops.pack_weight(eye), D, row_scale_shift=ss).double()   # W = I: out = x_hat
    xd = x.double()
    depth = 2 + -(-(D // 4) // 32) + 5
    mean, rstd, a, E_mean, _, E_rstd = _ln_bound(xd, xd.abs(), 0, depth, eps)
    want = a * rstd
    tol = rstd * E_mean + U * (mean * rstd).abs() + want.abs() * (E_rstd + 2.0 ** -20) + U * want.abs()
    err = (got - want).abs()
    assert bool((err <= tol).all()), f"prologue off by {float(err.max()):.3g}, worst / bound {float((err / tol).max()):.3g}"
    row_err = err.amax(1)
    ratio_ok = ratios <= 10
    assert float(row_err[ratio_ok].max()) <= 1e-4
    # the bound is what it says: (depth + 2) 2^-24 |mean| rstd, plus O(1e-5) from |x_hat| <~ 5
    assert bool((tol.amax(1) <= (depth + 3) * U * (mean * rstd).abs()[:, 0] + 3e-5).all())


# ============================================================================================== 4. the fused encoder
def _encoder_model(Dv, H, max_ctx_l, double_branch, seed):
    from dkd_b200.model import DLDKD
    cfg = ref_shim.model_config(Dv, 768, hidden=H, n_heads=4, max_ctx_l=max_ctx_l, max_desc_l=30)
    opt = ref_shim.options()
    opt.double_branch = double_branch
    torch.manual_seed(seed)
    m = DLDKD(cfg, opt).cuda().eval()
    with torch.no_grad():                       # non-trivial LayerNorm parameters and biases (reset_parameters: 1 / 0)
        for p in m.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    return m


def _dead_video_bounds(m64, b, x64, keep):
    """Propagate the fully-masked-attention bound of section 1 (weights good to expm1(2 GRID) relative, any fp32
    implementation) through the layers that follow it, per output, from float64 intermediates of the mirror:
    dense (|Wd|), residual + LayerNorm (|J| <= rstd |gamma| (I + 1 1^T / D + |a_hat| |a_hat|^T / D)), out mapping
    (|Wo|), key / value mappings.  Zero on videos with a valid frame."""
    from dkd_b200.encoder import FusedContextEncoder
    proj, pos, enc, outm, km, vm = FusedContextEncoder._branch_modules(m64, b)
    att, so = getattr(enc, "self"), enc.output
    B, L, _ = x64.shape
    X2 = pos(proj(x64))
    split = lambda t: t.view(B, L, att.heads, att.dh).transpose(1, 2)  # noqa: E731
    q, k, v = split(att.query(X2)), split(att.key(X2)), split(att.value(X2))
    p = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(att.dh), -1)      # a fully masked row: the raw scores
    e_ctx = math.expm1(2 * GRID) * (p @ v.abs()).transpose(1, 2).reshape(B, L, -1)
    e_ctx = e_ctx * (~keep.any(1)).double()[:, None, None]
    ctx = att(X2, keep.double()[:, None, :])
    z = so.dense(ctx) + X2
    e_dn = e_ctx @ so.dense.weight.abs().T
    rstd = 1.0 / torch.sqrt(z.var(-1, unbiased=False, keepdim=True) + so.LayerNorm.eps)
    ah = ((z - z.mean(-1, keepdim=True)) * rstd).abs()
    e_y = rstd * so.LayerNorm.weight.abs() * (e_dn + e_dn.mean(-1, keepdim=True) + ah * (ah * e_dn).mean(-1, keepdim=True))
    e_out = e_y @ outm.weight.abs().T
    return e_out, e_out @ km.weight.abs().T, e_out @ vm.weight.abs().T


ENCODER_CASES = [                   # Dv, H, branches, max_ctx_l, L, B, first video lengths (the rest random)
    (3072, 384, 2, 128, 128, 6, [128, 1, 0]),
    (3072, 128, 1, 32, 32, 4, [32, 1, 0]),
    (1024, 256, 2, 64, 64, 5, [64, 1, 0]),
    (1024, 512, 1, 128, 100, 3, [100, 1, 0]),
    (500, 128, 2, 64, 40, 4, [40, 1, 0]),
    (500, 384, 1, 32, 17, 3, [17, 0, 1]),
    (1024, 384, 2, 64, 1, 3, [1, 0, 1]),
    (3072, 512, 2, 32, 29, 1, [0]),
    (500, 256, 1, 128, 128, 1, [1]),
    (1024, 128, 2, 128, 77, 1, [77]),
    (500, 512, 2, 128, 128, 2, [128, 0]),
]


def _run_encoder_case(Dv, H, nb, max_ctx_l, L, B, lens0, seed):
    m = _encoder_model(Dv, H, max_ctx_l, nb == 2, seed)
    m64 = copy.deepcopy(m).double()                                 # the PyTorch mirror in float64
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, L, Dv, device="cuda", generator=g)
    x = x / (x.norm(dim=-1, keepdim=True) + 1e-5)
    lens = torch.randint(1, L + 1, (B,), device="cuda", generator=g)
    lens[:len(lens0)] = torch.tensor(lens0[:B], device="cuda")
    keep = torch.arange(L, device="cuda")[None] < lens[:, None]
    mask = keep.float()
    what = f"Dv={Dv} H={H} branches={nb} max_ctx_l={max_ctx_l} L={L} B={B}"
    with torch.no_grad():
        fused = m.enable_fused_encoder()._fused_encoder
        x64 = x.double()
        for msk in (mask, None):
            outs = fused.encode_context(x, msk, want_key_val=True)
            kv = outs[2]
            ref = m64.encode_context(x64, None if msk is None else msk.double())
            k_ = keep if msk is not None else torch.ones_like(keep)
            for b in range(nb):
                e_out, e_k, e_v = _dead_video_bounds(m64, b, x64, k_)
                kw, kb, vw, vb = m64.attention_params()[b]
                err = (outs[b].double() - ref[b]).abs()
                assert bool((err <= TOL + e_out).all()), (
                    f"{what} branch {b} mask={msk is not None}: off by {float(err.max()):.3g}")
                # the key / value mappings add their own K = H contraction to the 1e-4 of their input
                for got_kv, wk, bk, e in ((kv[b][0], kw, kb, e_k), (kv[b][1], vw, vb, e_v)):
                    want = torch.nn.functional.linear(ref[b], wk, bk)
                    assert bool(((got_kv.double() - want).abs() <= 2 * TOL + e).all()), f"{what} branch {b} key/value"
            if nb == 1:
                assert outs[1] is None and len(kv) == 1


@pytest.mark.parametrize("Dv,H,nb,max_ctx_l,L,B,lens0", ENCODER_CASES)
def test_fused_encoder_matches_float64_mirror(ops, dkd, Dv, H, nb, max_ctx_l, L, B, lens0):
    _run_encoder_case(Dv, H, nb, max_ctx_l, L, B, lens0, seed=Dv + H + L + B)


def test_fused_encoder_tvr_corpus_rows(ops, dkd):
    """2,179 videos x 128 frames x 3072-d, both branches: the production schedule of every GEMM."""
    _run_encoder_case(3072, 384, 2, 128, 128, 2179, [128, 1, 0], seed=2179)


# ---------------------------------------------------------------------------------------------- refusals
def _record_launches(monkeypatch):
    """Replace every C-ABI call by one that records its name and raises: a check that is missing reaches it."""
    from dkd_b200 import _lib
    calls = []

    def fake(name, *a):
        calls.append(name)
        raise RuntimeError(f"{name} reached a launch")
    monkeypatch.setattr(_lib, "call", fake)
    return calls


@pytest.mark.parametrize("max_ctx_l,L", [(32, 33), (64, 128), (32, 129), (160, 129)])
def test_encode_context_rejects_videos_longer_than_the_tables_before_any_launch(ops, dkd, monkeypatch, max_ctx_l, L):
    m = _encoder_model(64, 128, max_ctx_l, True, 0).enable_fused_encoder()
    x = torch.randn(2, L, 64, device="cuda")
    mask = torch.ones(2, L, device="cuda")
    calls = _record_launches(monkeypatch)
    with torch.no_grad():
        with pytest.raises(ValueError, match="frames per video"):
            m._fused_encoder.encode_context(x, mask)
    assert calls == []


def test_layernorm_rows_rejects_short_or_wrong_width_position_table(ops, monkeypatch):
    x = torch.randn(20, 64, device="cuda")
    gamma, beta = torch.ones(64, device="cuda"), torch.zeros(64, device="cuda")
    calls = _record_launches(monkeypatch)
    for pos, L in ((torch.randn(9, 64, device="cuda"), 10), (torch.randn(10, 68, device="cuda"), 10),
                   (torch.randn(10, 60, device="cuda"), 10)):
        with pytest.raises(ValueError, match="pos"):
            ops.layernorm_rows(x, gamma, beta, 1e-5, pos=pos, L=L)
    assert calls == []


@pytest.mark.parametrize("H,heads,limit", [(160, 4, "head size 40"), (48, 3, "multiple of 32"),
                                           (640, 5, "at most 512"), (576, 4, "head size 144")])
def test_pack_rejects_shapes_the_kernels_cannot_run(ops, dkd, monkeypatch, H, heads, limit):
    from dkd_b200.model import DLDKD
    cfg = ref_shim.model_config(64, 64, hidden=H, n_heads=heads, max_ctx_l=32, max_desc_l=8)
    m = DLDKD(cfg, ref_shim.options()).cuda().eval()
    calls = _record_launches(monkeypatch)
    with pytest.raises(ValueError, match=limit):
        m.enable_fused_encoder()
    assert calls == []
