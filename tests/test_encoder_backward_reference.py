"""The backward's error bound (tests/_encoder_backward_reference.py) checked without a GPU against a float32 emulation of
crl_zone_encode_backward's algorithm: the honest emulation stays inside the bound for every summation order tried and a
truncating adder, with the rows cut into partials by the launch rule; each of a list of plausible kernel bugs lands
outside it for at least one shape of the grid.  The mutation table is printed (largest |err| / r over the grid)."""
import pytest
import torch

from tests import _encoder_backward_reference as bref
from tests import _encoder_reference as ref
from tests.test_encoder_reference import bf, fsum

# (N, h, obs_dim, zone_dim): both slot counts with and without padding, one and two M-blocks (h 126 / 129 .. 190), one
# and two K steps of layer 1 with and without its lo column
GRID = [(1, 1, 1, 1), (5, 14, 8, 7), (8, 31, 8, 8), (9, 129, 24, 6), (15, 185, 8, 6), (16, 190, 24, 7), (6, 160, 1, 14)]
B = 24
SMS = 2                  # two partials, several tiles each
ORDERS = ['seq', 'rev', 'perm', 'tree']


def make_case(N, h, obs_dim, Z, seed=0):
    g = torch.Generator().manual_seed(seed + 1000 * N + h)
    rn = lambda *s, scale=1.0: torch.randn(*s, generator=g) * scale
    w = {'w1': rn(h, obs_dim + Z, scale=0.4), 'b1': rn(h, scale=0.2), 'w2': rn(h, h, scale=1.5 / h ** 0.5),
         'b2': rn(h, scale=0.2)}
    return w, rn(B, obs_dim), rn(B, N, Z), rn(B, h), g


def emulate_backward(w, obs, zobs, gp, order='seq', rz=False, mut=None, gen=None):
    """The kernel's algorithm in fp32: {'dw1', 'db1', 'dw2', 'db2'}."""
    Bn, N, Z = zobs.shape
    h, in_dim = w['w1'].shape
    S = ref.slots_per_env(N)
    if mut == 'pad':                           # padding slots loaded as real rows (zero features, ones columns)
        zobs = torch.cat([zobs, torch.zeros(Bn, S - N, Z)], 1)
    n_rows = zobs.shape[1]
    x = bf(ref.zone_rows(obs, zobs).to(torch.float32))
    b1hi, b2hi = bf(w['b1']), bf(w['b2'])
    b1lo, b2lo = bf(w['b1'] - b1hi), bf(w['b2'] - b2hi)
    if not ref.has_l1_lo(in_dim):
        b1lo = torch.zeros_like(b1lo)
    W1, W2 = bf(w['w1']), bf(w['w2'])
    ex = lambda b: b.expand(Bn, n_rows, h)[..., None]
    acc1 = fsum(torch.cat([x[:, :, None, :] * W1, ex(b1hi), ex(b1lo)], -1), order, rz, gen=gen)
    h1 = bf(acc1.clamp_min(0.0))
    acc2 = fsum(torch.cat([h1[:, :, None, :] * W2, ex(b2hi), ex(b2lo)], -1), order, rz, gen=gen)
    g = gp.clone()
    inv = torch.tensor(1.0 if mut == 'no_inv_n' else 1.0 / N, dtype=torch.float32)
    d2 = bf(g * inv)[:, None, :].expand(Bn, n_rows, h).clone()
    if mut == 'neighbour':                     # env 1's last slot reads env 0's g
        d2[1, N - 1] = d2[0, N - 1]
    dh2 = d2 if mut == 'no_mask2' else torch.where(acc2 > 0, d2, torch.zeros_like(d2))
    W2t = W2.T if mut == 'w2_for_w2t' else W2  # terms[j][i] = W2[i][j] dH2[i]
    acc = fsum(dh2[:, :, None, :] * W2t.T[None, None], order, rz, gen=gen)
    dh1 = bf(acc) if mut == 'no_mask1' else torch.where(h1 > 0, bf(acc), torch.zeros_like(acc))
    ones = torch.ones(Bn, n_rows, 2)
    h1f = torch.cat([h1, ones], -1)            # the ones rows h, h + 1 of H1
    xf = torch.cat([x, ones if ref.has_l1_lo(in_dim) else ones[..., :1]], -1)
    # partials: tile t of TILE_ROWS / S envs goes to CTA t % grid
    per_tile = bref.TILE_ROWS // S
    grid, _ = bref.launch(Bn, N, SMS)
    tile_of = torch.arange(Bn) // per_tile
    parts2, parts1 = [], []
    for p in range(grid):
        sel = (tile_of % grid) == p
        a2 = dh2[sel].reshape(-1, h)
        a1 = dh1[sel].reshape(-1, h)
        parts2.append(fsum(a2[:, :, None] * h1f[sel].reshape(-1, h + 2)[:, None, :], order, rz, dim=0, gen=gen))
        parts1.append(fsum(a1[:, :, None] * xf[sel].reshape(-1, xf.shape[-1])[:, None, :], order, rz, dim=0, gen=gen))
    if mut == 'drop_partial':
        parts2, parts1 = parts2[1:], parts1[1:]
    if mut == 'twice_partial':
        parts2, parts1 = parts2 + parts2[:1], parts1 + parts1[:1]
    t2 = sum(p.double() for p in parts2).float()
    t1 = sum(p.double() for p in parts1).float()
    db2, db1 = t2[:, h], t1[:, in_dim]
    if mut == 'db_hi_lo':
        db2 = t2[:, h] + t2[:, h + 1]
        if ref.has_l1_lo(in_dim):
            db1 = t1[:, in_dim] + t1[:, in_dim + 1]
    if mut == 'db2_row':
        db2 = t2[:, h - 1]                     # the last hidden row instead of the ones row
    return {'dw2': t2[:, :h], 'db2': db2, 'dw1': t1[:, :in_dim], 'db1': db1}


def _bound(w, obs, zobs, gp):
    return bref.backward_bound(w['w1'], w['b1'], w['w2'], w['b2'], obs, zobs, gp, SMS)


def _worst(out, want):
    return {k: ref.err_ratio(out[k], *want[k])[0] for k in want}


@pytest.mark.parametrize('shape', GRID, ids=lambda s: 'N%d-h%d-obs%d-Z%d' % s)
def test_honest_emulation_stays_inside_the_bound(shape):
    w, obs, zobs, gp, gen = make_case(*shape)
    want = _bound(w, obs, zobs, gp)
    worst = {}
    for order in ORDERS:
        for rz in (False, True):
            for k, v in _worst(emulate_backward(w, obs, zobs, gp, order, rz, gen=gen), want).items():
                worst[k] = max(worst.get(k, 0.0), v)
    print(shape, {k: round(v, 4) for k, v in worst.items()})
    assert all(v <= 1.0 for v in worst.values()), worst


MUTATIONS = ['no_inv_n', 'no_mask2', 'no_mask1', 'w2_for_w2t', 'neighbour', 'pad', 'db_hi_lo', 'db2_row',
             'drop_partial', 'twice_partial']


def test_each_mutation_lands_outside_the_bound():
    rows, missed = [], []
    for mut in MUTATIONS:
        worst = 0.0
        for shape in GRID:
            w, obs, zobs, gp, _ = make_case(*shape)
            worst = max(worst, max(_worst(emulate_backward(w, obs, zobs, gp, mut=mut), _bound(w, obs, zobs, gp)).values()))
        rows.append(f'{mut:14s} worst |err|/r {worst:10.3g} {"CAUGHT" if worst > 1 else "missed"}')
        if worst <= 1.0:
            missed.append(mut)
    print('\n' + '\n'.join(rows))
    assert not missed, missed


def test_the_bound_is_not_vacuous():
    """The radius is small against the values: a bound that is wide everywhere would pass any kernel.  (A few elements
    collect a wide term from a relu mask whose interval straddles 0; the typical radius is what is checked.  dW1 / db1
    carry the bf16 rounding of dH1, 2^-9 relative per term, so their typical radius is near 1e-3 of the largest value.)"""
    w, obs, zobs, gp, _ = make_case(*GRID[4])
    want = _bound(w, obs, zobs, gp)
    for k, (c, r) in want.items():
        assert float(r.median()) < 5e-3 * float(c.abs().max()), k


def test_launch_rule():
    assert bref.launch(1, 15, 148) == (1, 64)
    assert bref.launch(65536, 15, 148) == (148, 64 * 111)      # 16,384 tiles of 4 envs
    assert bref.launch(65536, 8, 148) == (148, 64 * 56)        # 8,192 tiles of 8 envs
    assert bref.launch(9, 8, 148) == (2, 64)
