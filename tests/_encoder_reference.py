"""A float64 reference of the zone encoder (csrc/crl_encode.cu) with a rigorous per-element error bound.

Every function returns a centre ``c`` and a radius ``r`` (float64 tensors of the output's shape) such that a correct
kernel gives ``|out - c| <= r`` in every element.  The bound models the arithmetic the kernels do, not a tolerance:

* Operands are rounded to bf16 (round to nearest even) from their fp32 values.  A product of two bf16 values has at
  most 16 significant bits, so it is exact in fp32 (and in float64 here).
* Accumulation is in fp32 (TMEM accumulators, the fp32 adds of the epilogues) with an unknown order and an unknown
  rounding mode: any summation tree of K terms makes K - 1 roundings, each at most one fp32 ulp (2^-23 relative, which
  covers round-to-nearest and truncating adders) of a partial sum whose magnitude is at most sum |terms|.  So a sum of
  K terms is within ``(K + 2) * 2^-23 * sum |terms|`` of the exact sum; the + 2 covers the second-order terms.  Adding
  an exact zero (padding rows, zero weights) makes no rounding.  A final product by fp32 ``1/N`` counts as one more
  rounding.  ``U`` is 2^-23 times (1 + 2^-20), which also covers the float64 rounding of the centre (K 2^-53 relative).
* Biases of the fast kernel ride in the GEMMs as bf16 hi = bf16(b) and lo = bf16(b - hi) terms multiplied by constant-1
  entries (pack_kernel).  Layer 1 carries the lo term only when ``in_dim + 1`` is not 16 or 32 (its padded K has no
  second spare column then); layer 2 and the head always carry it.  The ones entries of layer 2 are outputs of two
  generator rows of W1 (1 at the ones column, 0 elsewhere): a non-finite input row makes them NaN (0 * inf), so the
  whole slot becomes NaN through the bias terms.  ``_nan_of_row`` reproduces that.
* ``h1 = bf16_rn(relu(acc1))`` is carried as an interval: relu and bf16 RN are monotone, so an accumulator inside
  ``[p - r, p + r]`` rounds to a value inside ``[bf16(relu(p - r)), bf16(relu(p + r))]``; when the bound straddles a
  rounding boundary both neighbours are allowed, and the spread goes on through ``|W2|``.
* Pooling is an fp32 sum over the env's real slots (padding rows are exactly 0 in the fast kernel and skipped in the
  precise one) times fp32 ``1/N`` (the rounded reciprocal, exactly as the kernels hold it).
* Head (crl_encoder_head): ``[obs, pooled, 1, 1]`` and the weights rounded to bf16, the bias as hi + lo, one fp32
  accumulation.  In the fused forward and in ``zone_embedding`` pooled is itself an interval; its bf16 image lies in
  the bf16 rounding of that interval (the fused path rounds the same fp32 value the two-call path would).
* Precise mode (crl_zone_encode_precise): each operand v is split into hi = bf16(v), lo = bf16(v - hi) (v - hi is exact
  in fp32), and a product is W_hi X_hi + W_lo X_hi + W_hi X_lo (the lo lo term is dropped), three MMAs into one
  accumulator.  The fp32 biases are added in the epilogue (one more rounded term).  For the layer-1 activation, an
  interval of v gives hi in the bf16 rounding of the interval and hi + lo within 2^-16 |v| of v (each bf16 rounding is
  within 2^-8 relative), so the three products equal W_hi (hi + lo) + W_lo hi with both factors bounded.  The precise
  head is the fast head kernel run three times, (W, X), (W - bf16 W, X), (W, X - bf16 X), and two fp32 adds.

The accumulation term dominates the radius: about 3e-4 of a pooled value at h = 185 for the fast kernel, and three
times that for the precise one, whose K counts all three products (its measured error is near 1e-6, so the precise
mode's tests keep their bar against the fp32 module beside this bound).

Non-finite inputs follow IEEE arithmetic in float64 (0 * inf = NaN, NaN through relu), so the reference is non-finite
exactly where a correct kernel's output is.  Compute on the kernel's device: B = 65,536 envs is a few float64 GEMMs.
"""
import torch

U = 2.0 ** -23 * (1.0 + 2.0 ** -20)
BF16_REL = 2.0 ** -8          # |v - bf16_rn(v)| <= 2^-8 |v|


def bf16(t):
    """bf16 round-to-nearest of fp32 values (float64 in, float64 out; a float64 value goes through fp32 first, which
    keeps the rounding monotone)."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def split(t):
    """The precise kernels' split of fp32 values: hi = bf16(v), lo = bf16(v - hi)."""
    t = t.to(torch.float64)
    hi = bf16(t)
    return hi, bf16(t - hi)


def inv_n(n):
    """The kernels' fp32 1 / N."""
    return float(torch.tensor(1.0 / n, dtype=torch.float32))


def slots_per_env(n):
    return 8 if n <= 8 else 16


def has_l1_lo(in_dim):
    """Layer 1 of the fast kernel carries the bias lo term unless its padded K has no second spare column."""
    return in_dim + 1 not in (16, 32)


def zone_rows(obs, zone_obs):
    """(B, N, obs_dim + Z) float64 input rows [obs[e], zone_obs[e][z]]."""
    B, N, _ = zone_obs.shape
    return torch.cat([obs.to(torch.float64)[:, None, :].expand(B, N, obs.shape[1]), zone_obs.to(torch.float64)], -1)


def _nan_of_row(x):
    """0 for a finite row, NaN for a row with a non-finite entry (what 0 * x gives in a generator row)."""
    return (x * 0.0).sum(-1, keepdim=True)


def _relu_bf16_interval(p, r):
    return bf16((p - r).clamp_min(0.0)), bf16((p + r).clamp_min(0.0))


def _pool(lo, hi, n):
    """fp32 sum of the N slot intervals (B, N, h) times fp32 1/N -> centre, radius of pooled (B, h)."""
    k = inv_n(n)
    s_lo, s_hi = lo.sum(1), hi.sum(1)
    return (s_lo + s_hi) * (0.5 * k), (s_hi - s_lo) * (0.5 * k) + (n + 3) * U * k * s_hi


def pooled_bound(w1, b1, w2, b2, obs, zone_obs):
    """crl_zone_encode: pooled[e] = 1/N sum_z relu(L2(relu(L1([obs[e], zone_obs[e][z]]))))."""
    h, in_dim = w1.shape
    x = bf16(zone_rows(obs, zone_obs))
    W1, W2 = bf16(w1.to(torch.float64)), bf16(w2.to(torch.float64))
    b1hi, b1lo = split(b1)
    b2hi, b2lo = split(b2)
    if not has_l1_lo(in_dim):
        b1lo = torch.zeros_like(b1lo)
    p1 = x @ W1.T + (b1hi + b1lo)
    a1 = x.abs() @ W1.abs().T + (b1hi.abs() + b1lo.abs())
    lo1, hi1 = _relu_bf16_interval(p1, (in_dim + 2 + 2) * U * a1)
    g = 1.0 + _nan_of_row(x)                              # layer 2's ones entries
    p2 = ((lo1 + hi1) * 0.5) @ W2.T + (b2hi + b2lo) * g
    a2 = hi1 @ W2.abs().T + (b2hi.abs() + b2lo.abs()) * g
    r2 = ((hi1 - lo1) * 0.5) @ W2.abs().T + (h + 2 + 2) * U * a2
    lo2, hi2 = (p2 - r2).clamp_min(0.0), (p2 + r2).clamp_min(0.0)
    return _pool(lo2, hi2, zone_obs.shape[1])


def _split_interval(lo, hi):
    """For v in [lo, hi] (lo >= 0): intervals of hi(v) = bf16(v) and of hi(v) + lo(v), as (lo, hi) pairs."""
    return (bf16(lo), bf16(hi)), (lo * (1.0 - BF16_REL ** 2), hi * (1.0 + BF16_REL ** 2))


def pooled_precise_bound(w1, b1, w2, b2, obs, zone_obs):
    """crl_zone_encode_precise."""
    h, in_dim = w1.shape
    N = zone_obs.shape[1]
    xh, xl = split(zone_rows(obs, zone_obs))
    W1h, W1l = split(w1)
    W2h, W2l = split(w2)
    b1, b2 = b1.to(torch.float64), b2.to(torch.float64)
    p1 = xh @ (W1h + W1l).T + xl @ W1h.T + b1
    a1 = xh.abs() @ (W1h.abs() + W1l.abs()).T + xl.abs() @ W1h.abs().T + b1.abs()
    r1 = (3 * in_dim + 1 + 2) * U * a1
    (hl, hh), (fl, fh) = _split_interval((p1 - r1).clamp_min(0.0), (p1 + r1).clamp_min(0.0))
    # W2_hi (hi + lo) + W2_lo hi, each factor an interval
    p2 = ((fl + fh) * 0.5) @ W2h.T + ((hl + hh) * 0.5) @ W2l.T + b2
    r2 = ((fh - fl) * 0.5) @ W2h.abs().T + ((hh - hl) * 0.5) @ W2l.abs().T
    a2 = hh @ (W2h.abs() + W2l.abs()).T + (2 * BF16_REL) * fh @ W2h.abs().T + b2.abs()
    r2 = r2 + (3 * h + 1 + 2) * U * a2
    return _pool((p2 - r2).clamp_min(0.0), (p2 + r2).clamp_min(0.0), N)


def _head_operands(obs, pooled_lo, pooled_hi):
    """bf16 interval of the head's input rows [obs, pooled] (pooled >= 0)."""
    o = bf16(obs.to(torch.float64))
    return torch.cat([o, bf16(pooled_lo)], -1), torch.cat([o, bf16(pooled_hi)], -1)


def head_bound(w, b, obs, pooled_lo, pooled_hi=None):
    """crl_encoder_head on [obs, pooled] with the weights (h, obs_dim + h) and bias (h,) it packed; pooled exact
    (pooled_hi None: the kernel's own fp32 pooled) or an interval (the fused forward, zone_embedding)."""
    if pooled_hi is None:
        pooled_hi = pooled_lo
    xl, xh = _head_operands(obs, pooled_lo.to(torch.float64), pooled_hi.to(torch.float64))
    W = bf16(w.to(torch.float64))
    bhi, blo = split(b)
    g = 1.0 + _nan_of_row(xh)                             # 0 * a non-finite input in the zero weights of [0 | W3]
    c = ((xl + xh) * 0.5) @ W.T + (bhi + blo) * g
    a = torch.maximum(xl.abs(), xh.abs()) @ W.abs().T + (bhi.abs() + blo.abs())
    r = ((xh - xl) * 0.5) @ W.abs().T + (w.shape[1] + 2 + 2) * U * a
    return c, r


def head_precise_bound(w, b, obs, pooled_lo, pooled_hi):
    """ZoneEncoder._head_precise: the head kernel on (W, X), (W - bf16 W, X) and (W, X - bf16 X), summed in fp32;
    pooled an interval."""
    obs = obs.to(torch.float64)
    oh, ol = split(obs)
    (ph_l, ph_h), (pf_l, pf_h) = _split_interval(pooled_lo.to(torch.float64), pooled_hi.to(torch.float64))
    Wh, Wl = split(w)
    bhi, blo = split(b)
    k = w.shape[1]
    # W_hi (hi + lo) + W_lo hi: the obs part is exact, the pooled part two intervals
    xf_l, xf_h = torch.cat([oh + ol, pf_l], -1), torch.cat([oh + ol, pf_h], -1)
    xh_l, xh_h = torch.cat([oh, ph_l], -1), torch.cat([oh, ph_h], -1)
    c = ((xf_l + xf_h) * 0.5) @ Wh.T + ((xh_l + xh_h) * 0.5) @ Wl.T + bhi + blo
    r = ((xf_h - xf_l) * 0.5) @ Wh.abs().T + ((xh_h - xh_l) * 0.5) @ Wl.abs().T
    xa = torch.maximum(xh_l.abs(), xh_h.abs())
    a = xa @ (Wh.abs() + Wl.abs()).T + (2 * BF16_REL) * xa @ Wh.abs().T + bhi.abs() + blo.abs()
    return c, r + (k + 2 + 2 + 2) * U * a


def interval(c, r):
    return c - r, c + r


def err_ratio(out, c, r):
    """Largest |out - c| / r over the elements where the reference is finite (0 if there are none), and whether
    ``out`` is non-finite exactly where the reference is."""
    out = out.to(torch.float64)
    fin = torch.isfinite(c)
    same = bool(torch.equal(torch.isfinite(out), fin))
    if not bool(fin.any()):
        return 0.0, same
    d = (out - c).abs()[fin]
    rr = r[fin]
    ratio = torch.where(d == 0, torch.zeros_like(d), d / rr)     # inf where the bound is exact (r = 0) and missed
    return float(ratio.max()), same
