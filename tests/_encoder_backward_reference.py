"""A float64 reference of the zone encoder's backward (crl_zone_encode_backward, csrc/crl_encode.cu) with a per-element
error bound: for every element of dW1, db1, dW2, db2 a centre ``c`` and a radius ``r`` such that a correct kernel gives
``|out - c| <= r``.  It reuses the forward's model (tests/_encoder_reference.py) and adds:

* The recomputed forward is the forward kernel's: h1 = bf16(relu(acc1)) as a bf16 interval, acc2 (the layer-2
  pre-activation, biases folded as bf16 hi + lo) as an interval.
* Relu masks.  mask2 = acc2 > 0 and mask1 = h1 > 0 are certain when the interval lies on one side of 0; when it
  straddles 0 both choices are allowed (the gradient element is the hull of 0 and its value).  A NaN pre-activation
  makes the mask 0, as the kernel's comparison does (select semantics: a masked-off NaN g gives 0).
* dH2 = mask2 ? bf16(fp32(g * fp32(1/N))) : 0 is computed exactly (fp32 product in float32, then bf16).
* dH1 = mask1 ? bf16(sum_i W2[i][j] dH2[i]) : 0: an fp32 sum of h terms, (h + 2) U sum|terms|, then the bf16 rounding
  of the interval (monotone).
* dW2 = sum_m dH2[m]^T [h1[m], 1], dW1 = sum_m dH1[m]^T [x[m], 1]: products of two intervals (mid-rad arithmetic),
  fp32 sums of K terms per partial -- K = the rows of one partial by the documented launch rule -- then the partials
  summed in fp64 and rounded once to fp32: (K + 3) U sum|terms| + (P + 2) 2^-52 sum|terms|.  db2 is the column of the
  ones row h, db1 the column of the input ones column: one column each, never hi + lo.
* Padding slots are exact zeros in a correct kernel and absent here.
"""
import torch

from tests import _encoder_reference as ref

U = ref.U
TILE_ROWS = 64            # rows of one backward tile (4 envs of 16 slots, 8 of 8)


def launch(B, N, sms):
    """The launch rule of crl_zone_encode_backward: (number of partials, largest rows of one partial)."""
    per_tile = TILE_ROWS // ref.slots_per_env(N)
    tiles = -(-B // per_tile)
    grid = min(tiles, sms)
    return grid, TILE_ROWS * (-(-tiles // grid))


def _hull(one, zero, lo, hi):
    """Interval of mask ? v : 0 for v in [lo, hi], the mask certain 1 (one), certain 0 (zero) or either."""
    z = torch.zeros_like(lo)
    return (torch.where(one, lo, torch.where(zero, z, torch.minimum(z, lo))),
            torch.where(one, hi, torch.where(zero, z, torch.maximum(z, hi))))


def _forward_intervals(w1, b1, w2, b2, obs, zone_obs):
    """The recomputed forward of one chunk of envs: x (bf16), h1 interval (lo1, hi1), layer-2 ones entry, acc2 (p2, r2)."""
    h, in_dim = w1.shape
    x = ref.bf16(ref.zone_rows(obs, zone_obs))
    W1, W2 = ref.bf16(w1.to(torch.float64)), ref.bf16(w2.to(torch.float64))
    b1hi, b1lo = ref.split(b1)
    b2hi, b2lo = ref.split(b2)
    if not ref.has_l1_lo(in_dim):
        b1lo = torch.zeros_like(b1lo)
    p1 = x @ W1.T + (b1hi + b1lo)
    a1 = x.abs() @ W1.abs().T + (b1hi.abs() + b1lo.abs())
    lo1, hi1 = ref._relu_bf16_interval(p1, (in_dim + 2 + 2) * U * a1)
    g = 1.0 + ref._nan_of_row(x)
    p2 = ((lo1 + hi1) * 0.5) @ W2.T + (b2hi + b2lo) * g
    a2 = hi1 @ W2.abs().T + (b2hi.abs() + b2lo.abs()) * g
    r2 = ((hi1 - lo1) * 0.5) @ W2.abs().T + (h + 2 + 2) * U * a2
    return x, lo1, hi1, g, p2, r2, W2


def _prod_sum(alo, ahi, blo, bhi):
    """sum over rows of a^T b for a in [alo, ahi], b in [blo, bhi] ((R, p), (R, q) -> (p, q)): centre, radius of the
    exact sum, and sum |terms| (its largest value)."""
    ac, ar = (alo + ahi) * 0.5, (ahi - alo) * 0.5
    bc, br = (blo + bhi) * 0.5, (bhi - blo) * 0.5
    c = ac.T @ bc
    r = ac.abs().T @ br + ar.T @ bc.abs() + ar.T @ br
    s = (ac.abs() + ar).T @ (bc.abs() + br)
    return c, r, s


def backward_bound(w1, b1, w2, b2, obs, zone_obs, g, sms, chunk=8192):
    """{'dw1', 'db1', 'dw2', 'db2'} -> (centre, radius) for grad_pooled g (B, h) and a device with `sms` SMs."""
    h, in_dim = w1.shape
    B, N, _ = zone_obs.shape
    P, K = launch(B, N, sms)
    k = torch.tensor(ref.inv_n(N), dtype=torch.float32)
    dev = w1.device
    c2 = torch.zeros(h, h + 1, dtype=torch.float64, device=dev)
    r2_, s2 = torch.zeros_like(c2), torch.zeros_like(c2)
    c1 = torch.zeros(h, in_dim + 1, dtype=torch.float64, device=dev)
    r1_, s1 = torch.zeros_like(c1), torch.zeros_like(c1)
    for e0 in range(0, B, chunk):
        sl = slice(e0, min(B, e0 + chunk))
        x, lo1, hi1, ones2, p2, r2, W2 = _forward_intervals(w1, b1, w2, b2, obs[sl], zone_obs[sl])
        d2 = ref.bf16((g[sl].to(torch.float32) * k).to(torch.float64))[:, None, :].expand_as(p2)
        dlo, dhi = _hull((p2 - r2) > 0, ~((p2 + r2) > 0), d2, d2)
        # dH1 accumulator: sum_i W2[i][j] dH2[i]
        dc, dr = (dlo + dhi) * 0.5, (dhi - dlo) * 0.5
        acc_c = dc @ W2
        acc_r = dr @ W2.abs() + (h + 2) * U * (torch.maximum(dlo.abs(), dhi.abs()) @ W2.abs())
        blo, bhi = ref.bf16(acc_c - acc_r), ref.bf16(acc_c + acc_r)
        elo, ehi = _hull(lo1 > 0, ~(hi1 > 0), blo, bhi)
        rows = lambda t: t.reshape(-1, t.shape[-1])
        h1f_lo, h1f_hi = torch.cat([lo1, ones2], -1), torch.cat([hi1, ones2], -1)
        c, r, s = _prod_sum(rows(dlo), rows(dhi), rows(h1f_lo), rows(h1f_hi))
        c2 += c; r2_ += r; s2 += s
        xf = rows(torch.cat([x, torch.ones_like(x[..., :1])], -1))
        c, r, s = _prod_sum(rows(elo), rows(ehi), xf, xf)
        c1 += c; r1_ += r; s1 += s
    acc = (K + 3) * U + (P + 2) * 2.0 ** -52
    r2_ = r2_ + acc * s2
    r1_ = r1_ + acc * s1
    return {'dw2': (c2[:, :h], r2_[:, :h]), 'db2': (c2[:, h], r2_[:, h]),
            'dw1': (c1[:, :in_dim], r1_[:, :in_dim]), 'db1': (c1[:, in_dim], r1_[:, in_dim])}
