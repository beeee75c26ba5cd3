"""The encoder's error bound (tests/_encoder_reference.py) checked without a GPU, against float32 emulations of each
kernel's arithmetic: an honest emulation stays inside the bound for every summation order tried and for a truncating
adder, and each of a list of plausible kernel bugs lands outside it for at least one shape of the grid.

The emulations do what the kernels do: bf16 operands (exact products), fp32 sums in a chosen order with round to
nearest or toward zero, the bias hi / lo terms, bf16 h1, the fp32 pool over real slots times fp32 1/N, the head over
bf16 [obs, pooled, 1, 1]; the precise kernel's split operands, three products and fp32 epilogue biases.  The mutation
table is printed with each mutation's verdict under the previous global bar (1e-3 of the largest L3(pooled); 1e-4
for the precise mode) and under the bound (largest |err| / r over the grid).
"""
import pytest
import torch

from tests import _encoder_reference as ref

# (N, h, obs_dim, zone_dim): every slots_per_env class and padding count, M-block 1 (h > 126), the largest h (190),
# one- and two-K-step layer 1 with and without the layer-1 lo column (in_dim 2, 14, 15, 16, 30, 31)
GRID = [(1, 1, 1, 1), (5, 14, 8, 7), (7, 31, 8, 8), (8, 126, 8, 6), (9, 129, 24, 6), (15, 185, 8, 6),
        (16, 190, 24, 7), (6, 160, 1, 14), (16, 189, 8, 8)]
B = 24
ORDERS = ['seq', 'rev', 'perm', 'tree']


def _rz(s):
    """float64 -> fp32 rounded toward zero."""
    r = s.to(torch.float32)
    over = r.to(torch.float64).abs() > s.abs()
    return torch.where(over, torch.nextafter(r, torch.zeros_like(r)), r)


def _add(a, b, rz):
    return _rz(a.to(torch.float64) + b.to(torch.float64)) if rz else a + b


def fsum(t, order, rz, dim=-1, gen=None):
    """fp32 sum of the terms along `dim`, one fp32 add at a time in the given order."""
    t = t.movedim(dim, 0).to(torch.float32)
    k = t.shape[0]
    if order == 'tree':
        while t.shape[0] > 1:
            if t.shape[0] % 2:
                t = torch.cat([t, torch.zeros_like(t[:1])])
            t = _add(t[0::2], t[1::2], rz)
        return t[0]
    idx = {'seq': range(k), 'rev': range(k - 1, -1, -1)}.get(order)
    if idx is None:
        idx = torch.randperm(k, generator=gen).tolist()
    acc = torch.zeros_like(t[0])
    for i in idx:
        acc = _add(acc, t[i], rz)
    return acc


def bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def bf_rz(t):
    """bf16 rounded toward zero (fp32 bits with the low half cleared)."""
    return (t.to(torch.float32).view(torch.int32) & ~0xffff).view(torch.float32)


def _rows(obs, zobs):
    return ref.zone_rows(obs, zobs).to(torch.float32)


def emulate_pooled(w, obs, zobs, order='seq', rz=False, mut=None, gen=None):
    """The fast zone kernel in fp32: (B, h) pooled."""
    Bn, N, _ = zobs.shape
    h, in_dim = w['w1'].shape
    x = _rows(obs, zobs)
    if mut == 'neighbour':                     # env 1's last slot reads env 0's
        x[1, N - 1] = x[0, N - 1]
    x = bf(x)
    b1hi, b2hi = bf(w['b1']), bf(w['b2'])
    b1lo, b2lo = bf(w['b1'] - b1hi), bf(w['b2'] - b2hi)
    if not ref.has_l1_lo(in_dim) or mut == 'no_l1_lo':
        b1lo = torch.zeros_like(b1lo)
    if mut == 'no_l2_lo':
        b2lo = torch.zeros_like(b2lo)
    t1 = torch.cat([x[:, :, None, :] * bf(w['w1']), b1hi.expand(Bn, N, h)[..., None], b1lo.expand(Bn, N, h)[..., None]], -1)
    a1 = fsum(t1, order, rz, gen=gen).clamp_min(0.0)
    h1 = bf_rz(a1) if mut == 'h1_rz' else bf(a1)
    t2 = torch.cat([h1[:, :, None, :] * bf(w['w2']), b2hi.expand(Bn, N, h)[..., None], b2lo.expand(Bn, N, h)[..., None]], -1)
    o = fsum(t2, order, rz, gen=gen).clamp_min(0.0)
    S = ref.slots_per_env(N)
    p = fsum(o, order, rz, dim=1, gen=gen) * torch.tensor(1.0 / (S if mut == 'inv_s' else N), dtype=torch.float32)
    if mut == 'unit':
        i = int(p.abs().argmax())
        p.view(-1)[i] *= 1.0 + 1e-3
    return p


def _split(t):
    hi = bf(t)
    return hi, bf(t - hi)


def emulate_pooled_precise(w, obs, zobs, order='seq', rz=False, mut=None, gen=None):
    """The precise zone kernel in fp32: split operands, three products, fp32 biases, the pool over real slots."""
    Bn, N, _ = zobs.shape
    xh, xl = _split(_rows(obs, zobs))
    w1h, w1l = _split(w['w1'])
    w2h, w2l = _split(w['w2'])
    kw = 0.0 if mut == 'no_w_lo' else 1.0
    kx = 0.0 if mut == 'no_x_lo' else 1.0

    def layer(xh, xl, wh, wl, b):
        t = torch.cat([xh[:, :, None, :] * wh, kw * xh[:, :, None, :] * wl, kx * xl[:, :, None, :] * wh], -1)
        return _add(fsum(t, order, rz, gen=gen), b.expand(t.shape[:-1]), rz).clamp_min(0.0)
    hh, hl = _split(layer(xh, xl, w1h, w1l, w['b1']))
    o = layer(hh, hl, w2h, w2l, w['b2'])
    if mut == 'pad_relu_b2':                   # padding slots counted as relu(b2)
        o = torch.cat([o, w['b2'].clamp_min(0.0).expand(Bn, ref.slots_per_env(N) - N, -1)], 1)
    return fsum(o, order, rz, dim=1, gen=gen) * torch.tensor(1.0 / N, dtype=torch.float32)


def emulate_head(wh, bh, obs, pooled, order='seq', rz=False, mut=None, gen=None):
    x = bf(torch.cat([obs, pooled.to(torch.float32)], -1))
    bhi = bf(bh)
    blo = torch.zeros_like(bhi) if mut == 'no_head_lo' else bf(bh - bhi)
    n, h = x.shape[0], bh.shape[0]
    t = torch.cat([x[:, None, :] * bf(wh), bhi.expand(n, h)[..., None], blo.expand(n, h)[..., None]], -1)
    return fsum(t, order, rz, gen=gen)


def emulate_head_precise(wh, bh, obs, pooled, order='seq', rz=False, gen=None):
    z = torch.zeros_like(bh)
    o = emulate_head(wh, bh, obs, pooled, order, rz, gen=gen)
    o = _add(o, emulate_head(wh - bf(wh), z, obs, pooled, order, rz, gen=gen), rz)
    return _add(o, emulate_head(wh, z, obs - bf(obs), pooled - bf(pooled), order, rz, gen=gen), rz)


def make_case(N, h, obs_dim, Z, seed=0):
    g = torch.Generator().manual_seed(seed + 1000 * N + h)
    rn = lambda *s, scale=1.0: torch.randn(*s, generator=g) * scale
    w = {'w1': rn(h, obs_dim + Z, scale=0.4), 'b1': rn(h, scale=0.2), 'w2': rn(h, h, scale=1.5 / h ** 0.5),
         'b2': rn(h, scale=0.2), 'w3': rn(h, h, scale=1.5 / h ** 0.5), 'b3': rn(h, scale=0.2),
         'wc': rn(h, obs_dim + h, scale=0.1), 'bc': rn(h, scale=0.1)}
    return w, rn(B, obs_dim), rn(B, N, Z), g


def bounds(w, obs, zobs):
    c, r = ref.pooled_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
    return c, r


def _head_weights(w, obs_dim):
    """[0 | W3], b3: zone_embedding's head."""
    return torch.cat([torch.zeros(w['w3'].shape[0], obs_dim), w['w3']], 1), w['b3']


@pytest.mark.parametrize('shape', GRID, ids=lambda s: 'N%d-h%d-obs%d-Z%d' % s)
def test_honest_emulations_stay_inside_the_bound(shape):
    N, h, obs_dim, Z = shape
    w, obs, zobs, g = make_case(*shape)
    c, r = bounds(w, obs, zobs)
    lo, hi = ref.interval(c, r)
    wh, bh = _head_weights(w, obs_dim)
    hc, hr = ref.head_bound(wh, bh, obs, lo, hi)
    worst = {}
    for order in ORDERS:
        for rz in (False, True):
            p = emulate_pooled(w, obs, zobs, order, rz, gen=g)
            worst['pooled'] = max(worst.get('pooled', 0.0), ref.err_ratio(p, c, r)[0])
            e = emulate_head(wh, bh, obs, p, order, rz, gen=g)
            worst['head(interval)'] = max(worst.get('head(interval)', 0.0), ref.err_ratio(e, hc, hr)[0])
            ec, er = ref.head_bound(wh, bh, obs, p)
            worst['head(own pooled)'] = max(worst.get('head(own pooled)', 0.0), ref.err_ratio(e, ec, er)[0])
            if obs_dim + Z <= 16:
                pc, pr = ref.pooled_precise_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
                pp = emulate_pooled_precise(w, obs, zobs, order, rz, gen=g)
                worst['precise'] = max(worst.get('precise', 0.0), ref.err_ratio(pp, pc, pr)[0])
                fc, fr = ref.head_precise_bound(w['wc'], w['bc'], obs, *ref.interval(pc, pr))
                fp = emulate_head_precise(w['wc'], w['bc'], obs, pp, order, rz, gen=g)
                worst['precise head'] = max(worst.get('precise head', 0.0), ref.err_ratio(fp, fc, fr)[0])
    print(shape, {k: round(v, 4) for k, v in worst.items()})
    assert all(v <= 1.0 for v in worst.values()), worst


def _l3(p, w):
    return p.to(torch.float64) @ w['w3'].double().T + w['b3'].double()


MUTATIONS = ['no_l1_lo', 'no_l2_lo', 'no_head_lo', 'inv_s', 'pad_relu_b2', 'h1_rz', 'unit', 'neighbour', 'no_w_lo',
             'no_x_lo']
PRECISE_MUTATIONS = ('pad_relu_b2', 'no_w_lo', 'no_x_lo')


def _mutation_ratios(mut, shape):
    """(largest |err| / r under the bound, largest err / bar under the previous global bar) for one shape."""
    N, h, obs_dim, Z = shape
    w, obs, zobs, g = make_case(*shape)
    if mut in PRECISE_MUTATIONS:
        if obs_dim + Z > 16:
            return None
        c, r = ref.pooled_precise_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
        p = emulate_pooled_precise(w, obs, zobs, mut=mut)
        exact = ref.zone_rows(obs, zobs)
        for i in (1, 2):
            exact = exact @ w[f'w{i}'].double().T + w[f'b{i}'].double()
            exact = exact.clamp_min(0.0)
        want = _l3(exact.mean(1), w)
        old = float((_l3(p, w) - want).abs().max()) / (1e-4 * max(1.0, float(want.abs().max())))
        return ref.err_ratio(p, c, r)[0], old
    c, r = bounds(w, obs, zobs)
    if mut == 'no_head_lo':
        wh, bh = _head_weights(w, obs_dim)
        hc, hr = ref.head_bound(wh, bh, obs, *ref.interval(c, r))
        e = emulate_head(wh, bh, obs, emulate_pooled(w, obs, zobs), mut=mut)
        old = float((e.double() - hc).abs().max()) / (1e-3 * max(1.0, float(hc.abs().max())))
        return ref.err_ratio(e, hc, hr)[0], old
    p = emulate_pooled(w, obs, zobs, mut=mut)
    want = _l3(c, w)
    old = float((_l3(p, w) - want).abs().max()) / (1e-3 * max(1.0, float(want.abs().max())))
    return ref.err_ratio(p, c, r)[0], old


def test_each_mutation_lands_outside_the_bound():
    rows, missed = [], []
    for mut in MUTATIONS:
        res = [x for x in (_mutation_ratios(mut, s) for s in GRID) if x is not None]
        new, old = max(x[0] for x in res), max(x[1] for x in res)
        rows.append(f'{mut:12s} bound: worst |err|/r {new:10.3g} {"CAUGHT" if new > 1 else "missed"}   '
                    f'previous bar: worst err/bar {old:8.3g} {"CAUGHT" if old > 1 else "missed"}')
        if new <= 1.0:
            missed.append(mut)
    print('\n' + '\n'.join(rows))
    assert not missed, missed


def test_the_bound_is_not_vacuous():
    """The radius is small against the values: a bound that is wide everywhere would pass any kernel."""
    w, obs, zobs, _ = make_case(*GRID[5])
    c, r = bounds(w, obs, zobs)
    assert float(r.max()) < 1e-3 * float(c.abs().max())
    pc, pr = ref.pooled_precise_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
    assert float(pr.max()) < 1e-3 * float(pc.abs().max())


def test_non_finite_rows_give_non_finite_envs():
    """A NaN zone row, an infinite obs: the reference says NaN for the whole env (the kernels' generator rows and
    split operands spread it), and every other env is untouched."""
    w, obs, zobs, _ = make_case(5, 14, 8, 7)
    c0, r0 = bounds(w, obs, zobs)
    zobs[3, 2, 4] = float('nan')
    obs[7, 1] = float('inf')
    for fn in (ref.pooled_bound, ref.pooled_precise_bound):
        c, r = fn(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
        bad = torch.zeros(B, dtype=torch.bool)
        bad[[3, 7]] = True
        assert bool(torch.isnan(c[bad]).all()) and bool(torch.isfinite(c[~bad]).all())
    c, r = ref.pooled_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs)
    assert torch.equal(c[~bad], c0[~bad]) and torch.equal(r[~bad], r0[~bad])
    hc, _ = ref.head_bound(w['wc'], w['bc'], obs, *ref.interval(c, r))
    assert bool(torch.isnan(hc[bad]).all()) and bool(torch.isfinite(hc[~bad]).all())
