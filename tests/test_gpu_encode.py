"""crl_zone_encode (tcgen05 kernel, csrc/crl_encode.cu) + the (B, h) third Linear = ZoneEnvModel's zone_net_
+ mean-pool (main/src/env_model.py:56-78; the mean commutes with the affine third layer).  The kernel multiplies bf16
operands with fp32 accumulation.  Two kinds of checks:
  against the float64 reference with a per-element error bound (tests/_encoder_reference.py): every element of
     pooled, of the head's output, of zone_embedding / forward and of the precise mode within its radius
     (|err| / r <= 1; the largest ratio per shape is printed);
  vs the REAL module's fp32 output (fixture) and vs torch fp32 ................... 1e-2 of the largest value
     (bf16 operand rounding through the two wide layers; measured 3e-3 .. 5e-3); precise mode: 1e-4
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from oracle import zone_model as zm  # noqa: E402
from tests import _encoder_reference as ref  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'model_zone_env.npz')
FP32_RTOL = 1e-2


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def _bound_of(sd, obs, zone_obs, precise=False):
    fn = ref.pooled_precise_bound if precise else ref.pooled_bound
    return fn(sd['zone_net_.0.weight'], sd['zone_net_.0.bias'], sd['zone_net_.2.weight'], sd['zone_net_.2.bias'], obs, zone_obs)


def _l3_weights(enc):
    return torch.cat([torch.zeros(enc.hidden, enc.obs_dim, device=enc.w3.device), enc.w3], 1), enc.b3


def _check(out, c, r, what, shape, ratios):
    ratio, same = ref.err_ratio(out, c, r)
    ratios[what] = ratio
    assert same, (what, shape, 'non-finite where the reference is finite, or the reverse')
    assert ratio <= 1.0, (what, shape, ratio)


def fp32_ref(sd, obs, zone_obs):
    B, N, _ = zone_obs.shape
    x = torch.cat([obs[:, None, :].expand(B, N, obs.shape[1]), zone_obs], dim=-1).to(torch.float64)
    for i in (0, 2, 4):
        x = x @ sd[f'zone_net_.{i}.weight'].to(torch.float64).T + sd[f'zone_net_.{i}.bias'].to(torch.float64)
        if i != 4:
            x = torch.relu(x)
    return (x.sum(dim=1) / N).to(torch.float32)


@pytest.mark.parametrize('tag,n', [('tsp', 15), ('cm', 6)])
def test_fixture_of_the_real_module(crl, tag, n):
    g = dict(np.load(GOLDEN))
    sd = {k[len(tag) + 4:]: torch.from_numpy(g[k]).cuda() for k in g if k.startswith(tag + '_sd_')}
    enc = crl.ZoneEncoder(sd, num_zones=n)
    obs, zobs = torch.from_numpy(g[f'{tag}_obs']).cuda(), torch.from_numpy(g[f'{tag}_zone_obs']).cuda()
    emb = enc.zone_embedding(obs, zobs)
    out = enc(obs, zobs)
    torch.cuda.synchronize()
    assert enc.healthy()
    c, r = _bound_of(sd, obs, zobs)
    w, b = _l3_weights(enc)
    e_twin, _ = ref.err_ratio(emb, *ref.head_bound(w, b, obs, *ref.interval(c, r)))
    e_fwd, _ = ref.err_ratio(out, *ref.head_bound(enc.fold_w, enc.fold_b, obs, *ref.interval(c, r)))
    e_emb = float(np.abs(emb.cpu().numpy() - g[f'{tag}_zone_emb']).max())
    e_out = float(np.abs(out.cpu().numpy() - g[f'{tag}_out']).max())
    scale = max(1.0, float(np.abs(g[f'{tag}_zone_emb']).max()))
    print(f'{tag}: |err|/r zone_emb {e_twin:.3f} forward {e_fwd:.3f}, vs real module zone_emb {e_emb:.2e}, forward {e_out:.2e}, scale {scale:.2f}')
    assert e_twin <= 1.0 and e_fwd <= 1.0 and e_emb <= FP32_RTOL * scale and e_out <= FP32_RTOL * scale
    # the numpy oracle agrees with what was compared against
    assert np.abs(zm.zone_embedding({k: v.cpu().numpy() for k, v in sd.items()}, g[f'{tag}_obs'], g[f'{tag}_zone_obs'])
                  - g[f'{tag}_zone_emb']).max() <= 2e-6


# (B, N, Z, h, D), D = per-env features (obs_dim).  The first six are ZoneEnvModel-like; the rest cover: N 1, 5, 7, 8,
# 9, 15, 16 (8- and 16-slot envs, 0..15 padding rows); h 1, 14, 31, 126 (ones rows end M-block 0), 129..190 (M-block 1;
# 190: its ones rows are the block's last two); in_dim 2, 14, 15 and 31 (no layer-1 lo column), 16 and 30 (two K
# steps); D 1, 8, 24, with D + h + 2 = 192 (head K exactly full) and 193; B = 1, envs per tile - 1 / exact / + 1 (16
# envs per tile for 8 slots, 8 for 16), 91 (the last tile is a CTA's second group), 65,536 (4,096 tiles: > 3 waves)
SHAPES = [(4099, 15, 6, 185, 8), (1, 15, 7, 185, 8), (777, 5, 6, 96, 8), (20000, 6, 7, 32, 8), (3001, 15, 7, 185, 10),
          (515, 6, 7, 64, 16),
          (1, 1, 1, 1, 1), (15, 5, 7, 14, 8), (16, 7, 8, 31, 8), (17, 8, 6, 126, 8), (7, 9, 6, 129, 24),
          (8, 16, 15, 160, 16), (9, 15, 6, 189, 8), (91, 16, 7, 189, 1), (3001, 5, 14, 190, 1), (515, 7, 7, 160, 24),
          (1000, 1, 22, 129, 8), (65536, 8, 6, 126, 8)]


def _weights(gen, h, in_dim, D):
    rn = lambda *s, scale=1.0: (torch.randn(*s, device='cuda', generator=gen) * scale)
    return {'zone_net_.0.weight': rn(h, in_dim, scale=0.4), 'zone_net_.0.bias': rn(h, scale=0.2),
            'zone_net_.2.weight': rn(h, h, scale=1.5 / h ** 0.5), 'zone_net_.2.bias': rn(h, scale=0.2),
            'zone_net_.4.weight': rn(h, h, scale=1.5 / h ** 0.5), 'zone_net_.4.bias': rn(h, scale=0.2),
            'combine_net_.weight': rn(h, D + h, scale=0.1), 'combine_net_.bias': rn(h, scale=0.1)}


def _nan_tail(t):
    """t as a view into a larger buffer that holds NaN past row B (a kernel reading rows >= B into valid outputs fails)."""
    buf = torch.full((t.shape[0] + 40,) + tuple(t.shape[1:]), float('nan'), device=t.device)
    buf[:t.shape[0]] = t
    return buf[:t.shape[0]]


class _Guarded:
    """An output (B, h) with guard rows of 7.0 on both sides."""
    def __init__(self, B, h):
        self.buf = torch.full((B + 6, h), 7.0, device='cuda')
        self.out = self.buf[3:B + 3]

    def intact(self):
        return bool((self.buf[:3] == 7.0).all()) and bool((self.buf[-3:] == 7.0).all())


@pytest.mark.parametrize('B,N,Z,h,D', SHAPES)
def test_random_batches_against_torch(crl, B, N, Z, h, D):
    """Every output of the encoder against the float64 reference's per-element bound, over a covering set of the
    shapes check_shape accepts: pooled (fast), the head on the kernel's own pooled, zone_embedding and forward (fused
    where the shape allows it, two calls otherwise), precise pooled and forward_precise (in_dim <= 16).  Inputs are
    views with NaN past row B, outputs have guard rows on both sides.  Also against torch fp32 (1e-2)."""
    gen = torch.Generator(device='cuda').manual_seed(B + h)
    sd = _weights(gen, h, D + Z, D)
    obs = _nan_tail(torch.randn(B, D, device='cuda', generator=gen))
    zobs = _nan_tail(torch.randn(B, N, Z, device='cuda', generator=gen))
    enc = crl.ZoneEncoder(sd, num_zones=N)
    shape, ratios = (B, N, Z, h, D), {}
    g = _Guarded(B, h)
    pooled = enc.pooled(obs, zobs, out=g.out)
    torch.cuda.synchronize()
    assert enc.healthy() and g.intact()
    c, r = _bound_of(sd, obs, zobs)
    _check(pooled, c, r, 'pooled', shape, ratios)
    lo, hi = ref.interval(c, r)
    ref32 = fp32_ref(sd, obs, zobs)
    emb = torch.nn.functional.linear(pooled, sd['zone_net_.4.weight'], sd['zone_net_.4.bias'])
    scale = max(1.0, float(ref32.abs().max()))
    assert float((emb - ref32).abs().max()) <= FP32_RTOL * scale
    # the head kernel on the kernel's own pooled: the folded forward and [0 | W3]
    l3_w, l3_b = _l3_weights(enc)
    for what, packed, w, b in (('head', enc.packed_head, enc.fold_w, enc.fold_b), ('head L3', enc.packed_l3, l3_w, l3_b)):
        g2 = _Guarded(B, h)
        out = enc._head(packed, obs, pooled, out=g2.out)
        torch.cuda.synchronize()
        assert g2.intact()
        _check(out, *ref.head_bound(w, b, obs, pooled), what, shape, ratios)
    # zone_embedding and forward: the fused two-kernel forward where the shape is ZoneEnvModel's own, else two calls
    fused = enc._workspace(B) is not None
    g3, g4 = _Guarded(B, h), _Guarded(B, h)
    emb_k = enc.zone_embedding(obs, zobs, out=g3.out)
    fwd_k = enc._forward(obs, zobs, out=g4.out)
    torch.cuda.synchronize()
    assert enc.healthy() and g3.intact() and g4.intact()
    _check(emb_k, *ref.head_bound(l3_w, l3_b, obs, lo, hi), 'zone_embedding', shape, ratios)
    _check(fwd_k, *ref.head_bound(enc.fold_w, enc.fold_b, obs, lo, hi), 'forward', shape, ratios)
    assert float((emb_k - ref32).abs().max()) <= FP32_RTOL * scale
    if D + Z <= 16:
        g5 = _Guarded(B, h)
        pp = enc.pooled_precise(obs, zobs, out=g5.out)
        fp = enc.forward_precise(obs, zobs)
        torch.cuda.synchronize()
        assert enc.healthy() and g5.intact()
        pc, pr = _bound_of(sd, obs, zobs, precise=True)
        _check(pp, pc, pr, 'precise', shape, ratios)
        _check(fp, *ref.head_precise_bound(enc.fold_w, enc.fold_b, obs, *ref.interval(pc, pr)), 'forward_precise', shape, ratios)
    print(f'B={B} N={N} Z={Z} h={h} D={D} ({"fused" if fused else "two-call"} forward): largest |err|/r ' +
          ', '.join(f'{k} {v:.3f}' for k, v in ratios.items()))
    # second call on the same encoder (barrier phases, TMEM re-allocation) gives the same bits
    assert torch.equal(enc.pooled(obs, zobs), pooled)


@pytest.mark.parametrize('N,Z', [(15, 6), (6, 7)])
def test_non_finite_inputs(crl, N, Z):
    """NaN in one zone row of the first env of a tile, of the last env of a tile and of the last env of the batch, +inf
    in one obs, and one env with |x| ~ 1e15: every other env is bit-identical to a clean run, and the affected envs are
    non-finite exactly where the float64 reference is (NaN: the whole env) and within the bound elsewhere.  Fast pooled,
    the fused forward, zone_embedding, precise pooled and forward_precise."""
    B, h = 3001, 185
    per_tile = 128 // ref.slots_per_env(N)
    gen = torch.Generator(device='cuda').manual_seed(11)
    sd = _weights(gen, h, 8 + Z, 8)
    obs = torch.randn(B, 8, device='cuda', generator=gen)
    zobs = torch.rand(B, N, Z, device='cuda', generator=gen)
    enc = crl.ZoneEncoder(sd, num_zones=N)
    assert enc._workspace(B) is not None                       # the fused forward runs
    runs = lambda o, z: {'pooled': enc.pooled(o, z), 'forward': enc(o, z), 'zone_embedding': enc.zone_embedding(o, z),
                         'precise': enc.pooled_precise(o, z), 'forward_precise': enc.forward_precise(o, z)}
    clean = runs(obs, zobs)
    nan_envs = [2 * per_tile, 3 * per_tile - 1, B - 1]
    o2, z2 = obs.clone(), zobs.clone()
    for k, e in enumerate(nan_envs):
        z2[e, (k * 5) % N, k % Z] = float('nan')
    inf_env, big_env = 40, 50
    o2[inf_env, 3] = float('inf')
    o2[big_env] *= 1e15
    z2[big_env] *= 1e15
    dirty = runs(o2, z2)
    torch.cuda.synchronize()
    assert enc.healthy()
    hit = torch.zeros(B, dtype=torch.bool, device='cuda')
    hit[nan_envs + [inf_env, big_env]] = True
    c, r = _bound_of(sd, o2, z2)
    pc, pr = _bound_of(sd, o2, z2, precise=True)
    l3_w, l3_b = _l3_weights(enc)
    want = {'pooled': (c, r), 'forward': ref.head_bound(enc.fold_w, enc.fold_b, o2, *ref.interval(c, r)),
            'zone_embedding': ref.head_bound(l3_w, l3_b, o2, *ref.interval(c, r)), 'precise': (pc, pr),
            'forward_precise': ref.head_precise_bound(enc.fold_w, enc.fold_b, o2, *ref.interval(pc, pr))}
    ratios = {}
    for k in clean:
        assert torch.equal(dirty[k][~hit], clean[k][~hit]), k
        wc, wr = want[k]
        assert bool(torch.isnan(wc[nan_envs + [inf_env]]).all()) and bool(torch.isfinite(wc[big_env]).all())
        _check(dirty[k][hit], wc[hit], wr[hit], k, (N, Z), ratios)
    print(f'N={N}: affected envs, largest |err|/r ' + ', '.join(f'{k} {v:.3f}' for k, v in ratios.items()))


def test_encoder_on_the_env_outputs(crl):
    """The fused step's outputs feed the encoder directly (obs (B,8), zone_obs (B,N,Z) as CrlOut lays them out)."""
    g = dict(np.load(GOLDEN))
    sd = {k[7:]: torch.from_numpy(g[k]).cuda() for k in g if k.startswith('tsp_sd_')}
    env = crl.ZoneVecEnv('PointTSP-v0', 4096)
    env.seed(3)
    obs = env.reset()
    for _ in range(5):
        obs, *_ = env.step_random(action_seed=2)
    enc = crl.ZoneEncoder(sd, num_zones=15)
    y = enc(obs)
    ref = torch.nn.functional.linear(torch.cat([obs['obs'], fp32_ref(sd, obs['obs'], obs['zone_obs'])], -1),
                                     sd['combine_net_.weight'], sd['combine_net_.bias'])
    assert enc.healthy() and y.shape == (4096, 185)
    assert float((y - ref).abs().max()) <= FP32_RTOL * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize('env_id', ['PointTSP-v0', 'PointTTSP-v0', 'ColourMatch-v0', 'PointTSP-v1', 'PointTTSP-v3',
                                    'PointTTSP-v1', 'PointTSP-v3', 'ColourMatch-v3', 'PointTSP-v4', 'PointTSP-v5',
                                    'zone-goals/PointTSP-v4', 'zone-goals/PointTSP-v5', 'walled/PointTSP-v0',
                                    'walled/PointTSP-v1', 'walled/PointTTSP-v0', 'walled/PointTTSP-v1',
                                    'walled/ColourMatch-v0'])
def test_rows_built_from_the_state_planes_are_the_rows_the_step_writes(crl, env_id):
    """crl_zone_encode_state builds the zone part of the encoder's input from the state planes (zone centres,
    visited / colour bits, timeouts, cooldowns, step count).  It must see bit for bit the rows the step writes to
    zone_obs -- so `pooled` is bit-identical between the two paths -- also for envs that have visited zones, run
    cooldowns, been reset; and a rollout with env.write_zone_obs = False (CRL_STEP_NO_ZONE_OBS: the step neither
    builds nor writes zone_obs) gives the same embeddings as one that materialises them."""
    B, h = 3000, 96
    N, Z = crl.ENV_SPECS[env_id].num_zones, crl.ENV_SPECS[env_id].zone_dim
    gen = torch.Generator(device='cuda').manual_seed(5)
    rn = lambda *s_, scale=1.0: (torch.randn(*s_, device='cuda', generator=gen) * scale)
    sd = {'zone_net_.0.weight': rn(h, 8 + Z, scale=0.4), 'zone_net_.0.bias': rn(h, scale=0.2),
          'zone_net_.2.weight': rn(h, h, scale=0.15), 'zone_net_.2.bias': rn(h, scale=0.2),
          'zone_net_.4.weight': rn(h, h, scale=0.15), 'zone_net_.4.bias': rn(h, scale=0.2),
          'combine_net_.weight': rn(h, 8 + h, scale=0.1), 'combine_net_.bias': rn(h, scale=0.1)}
    enc = crl.ZoneEncoder(sd, num_zones=N)
    full, lean = crl.ZoneVecEnv(env_id, B), crl.ZoneVecEnv(env_id, B)
    for e in (full, lean):
        e.seed(77)
        e.cfg.num_steps = 60                                   # short episodes: auto-resets inside the test
        e.reset()
    lean.write_zone_obs = False
    frozen = lean.zone_obs.clone()
    rs = np.random.RandomState(2)
    for t in range(90):
        a = torch.from_numpy(rs.uniform(-1, 1, (B, 2)).astype(np.float32)).cuda()
        if t % 7 == 3:                                         # zone events: visited bits / colour cycles / cooldowns
            z = int(rs.randint(N))
            for e in (full, lean):
                e.pose[t % 5::5, :2] = e.zone_xy[z, t % 5::5, :]
        full.step(a)
        lean.step(a)
        if t % 9 == 0 or t > 84:
            want = enc.pooled(full.obs, full.zone_obs)
            assert torch.equal(enc.pooled_from_state(full), want), (env_id, t)      # same env, both paths
            assert torch.equal(enc.pooled_from_state(lean), want), (env_id, t)      # the env that never wrote zone_obs
            assert torch.equal(enc.forward_from_state(lean), enc(full.obs, full.zone_obs)), (env_id, t)
    torch.cuda.synchronize()
    assert enc.healthy()
    assert torch.equal(lean.zone_obs, frozen)                  # CRL_STEP_NO_ZONE_OBS: untouched since the reset
    # aux is compared as bits: its .w word holds step count and visited mask, which can read as NaN in float32
    # (the hard instances' zones start visited)
    assert torch.equal(lean.obs, full.obs) and torch.equal(lean.result, full.result)
    assert torch.equal(lean.aux.view(torch.int32), full.aux.view(torch.int32))
    assert full.counters()['episodes'] == lean.counters()['episodes'] >= B


def test_unsupported_shapes_are_refused(crl):
    from combinatorial_rl_tasks_b200 import _lib
    import ctypes
    lib = _lib.load()
    n = ctypes.c_int64()
    assert lib.crl_encoder_packed_bytes(_lib.CrlEncoderShape(8, 6, 185, 15), ctypes.byref(n)) == 0 and n.value == 256 * 192 * 2 + 256 * 32
    assert lib.crl_encoder_packed_bytes(_lib.CrlEncoderShape(8, 6, 256, 15), ctypes.byref(n)) == -4    # two resident weights do not fit
    assert lib.crl_encoder_packed_bytes(_lib.CrlEncoderShape(20, 12, 64, 15), ctypes.byref(n)) == -2     # no room for the ones column in the 32-wide input
    assert lib.crl_encoder_head_packed_bytes(_lib.CrlEncoderShape(8, 6, 185, 15), ctypes.byref(n)) == 0 and n.value == 256 * 208 * 2
    # the edges of what check_shape accepts: h 190, N 16, in_dim 31, precise in_dim 16
    S = _lib.CrlEncoderShape
    for ok in (S(8, 6, 190, 15), S(8, 6, 185, 16), S(24, 7, 64, 15), S(1, 30, 64, 1)):
        assert lib.crl_encoder_packed_bytes(ok, ctypes.byref(n)) == 0, (ok.obs_dim, ok.zone_dim, ok.hidden, ok.num_zones)
    assert lib.crl_encoder_precise_packed_bytes(S(8, 8, 185, 15), ctypes.byref(n)) == 0
    # and one past each: h 191 (K of layer 2 > 192), N 0 and 17, in_dim 32, precise in_dim 17
    assert lib.crl_encoder_packed_bytes(S(8, 6, 191, 15), ctypes.byref(n)) == -4
    assert lib.crl_encoder_packed_bytes(S(8, 6, 185, 0), ctypes.byref(n)) == -2
    assert lib.crl_encoder_packed_bytes(S(8, 6, 185, 17), ctypes.byref(n)) == -2
    assert lib.crl_encoder_packed_bytes(S(24, 8, 64, 15), ctypes.byref(n)) == -2
    assert lib.crl_encoder_precise_packed_bytes(S(8, 9, 185, 15), ctypes.byref(n)) == -4
    # num_envs = 0: refused by every launch (non-null dummy pointers, so the batch size is what is refused)
    p = torch.zeros(1 << 16, dtype=torch.uint8, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    ptr, st, s0 = p.data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream
    shape = S(8, 6, 185, 15)
    assert lib.crl_zone_encode(shape, 0, ptr, ptr, ptr, ptr, st, s0) == -2
    assert lib.crl_zone_encode_precise(shape, 0, ptr, ptr, ptr, ptr, st, s0) == -2
    assert lib.crl_encoder_head(shape, 0, ptr, ptr, ptr, ptr, st, s0) == -2
    assert lib.crl_encoder_workspace_bytes(shape, 0, ctypes.byref(n)) == -2
    torch.cuda.synchronize()
    assert int(status.item()) == 0


@pytest.mark.parametrize('env_id,B,h', [('PointTSP-v0', 4099, 185), ('ColourMatch-v0', 1000, 185), ('PointTTSP-v0', 129, 185),
                                        ('PointTSP-v1', 77, 185), ('PointTSP-v0', 3000, 100), ('PointTTSP-v0', 2000, 64),
                                        ('ColourMatch-v0', 900, 127), ('PointTSP-v0', 1500, 33)])
def test_fused_forward_is_the_two_call_forward(crl, env_id, B, h):
    """crl_encoder_forward (the zone kernel writes the head kernel's bf16 operand image, no fp32 pooled in between, one
    bulk copy per 128 envs in the head) gives bit for bit what crl_zone_encode + crl_encoder_head give -- the head rounds
    pooled to bf16 either way -- from the materialised zone_obs and from the state planes; ragged batches; hidden widths
    whose last warp reaches beyond the image's width (100, 33), one M-block (64, 100) and two (127: the ones rows, 185)."""
    N, Z = crl.ENV_SPECS[env_id].num_zones, crl.ENV_SPECS[env_id].zone_dim
    gen = torch.Generator(device='cuda').manual_seed(B)
    rn = lambda *s_, scale=1.0: (torch.randn(*s_, device='cuda', generator=gen) * scale)
    sd = {'zone_net_.0.weight': rn(h, 8 + Z, scale=0.4), 'zone_net_.0.bias': rn(h, scale=0.2),
          'zone_net_.2.weight': rn(h, h, scale=0.1), 'zone_net_.2.bias': rn(h, scale=0.2),
          'zone_net_.4.weight': rn(h, h, scale=0.1), 'zone_net_.4.bias': rn(h, scale=0.2),
          'combine_net_.weight': rn(h, 8 + h, scale=0.1), 'combine_net_.bias': rn(h, scale=0.1)}
    enc = crl.ZoneEncoder(sd, num_zones=N)
    env = crl.ZoneVecEnv(env_id, B)
    env.seed(5)
    obs = env.reset()
    for _ in range(30):
        obs, *_ = env.step_random(action_seed=2)
    two = enc._head(enc.packed_head, obs['obs'], enc.pooled(obs['obs'], obs['zone_obs']))
    guard = torch.full((B + 2, h), 7.0, device='cuda')
    fused = enc._forward(obs['obs'], obs['zone_obs'], out=guard[:B])
    from_state = enc.forward_from_state(env)
    torch.cuda.synchronize()
    assert enc.healthy() and enc._workspace(B) is not None
    assert torch.equal(fused, two) and torch.equal(from_state, two)
    assert bool((guard[B:] == 7.0).all()) and bool(torch.isfinite(fused).all())


PRECISE_RTOL = 1e-4       # the like-for-like bar against the fp32 module (VERDICT r1 next #4); measured ~1e-5


@pytest.mark.parametrize('tag,n', [('tsp', 15), ('cm', 6)])
def test_precise_mode_against_the_real_modules_fp32_output(crl, tag, n):
    """crl_zone_encode_precise (split-bf16 operands, three MMAs per product, fp32 biases) against the fixture recorded
    from the REAL ZoneEnvModel in fp32: zone_emb and forward within 1e-4 of the largest value."""
    g = dict(np.load(GOLDEN))
    sd = {k[len(tag) + 4:]: torch.from_numpy(g[k]).cuda() for k in g if k.startswith(tag + '_sd_')}
    enc = crl.ZoneEncoder(sd, num_zones=n)
    torch.backends.cuda.matmul.allow_tf32 = False
    obs, zobs = torch.from_numpy(g[f'{tag}_obs']).cuda(), torch.from_numpy(g[f'{tag}_zone_obs']).cuda()
    emb = enc.zone_embedding_precise(obs, zobs)
    out = enc.forward_precise(obs, zobs)
    torch.cuda.synchronize()
    assert enc.healthy()
    e_emb = float(np.abs(emb.cpu().numpy() - g[f'{tag}_zone_emb']).max()) / max(1.0, float(np.abs(g[f'{tag}_zone_emb']).max()))
    e_out = float(np.abs(out.cpu().numpy() - g[f'{tag}_out']).max()) / max(1.0, float(np.abs(g[f'{tag}_out']).max()))
    e_fast = float(np.abs(enc(obs, zobs).cpu().numpy() - g[f'{tag}_out']).max()) / max(1.0, float(np.abs(g[f'{tag}_out']).max()))
    print(f'{tag}: precise zone_emb {e_emb:.2e}, forward {e_out:.2e} (fast bf16 forward {e_fast:.2e})')
    assert e_emb <= PRECISE_RTOL and e_out <= PRECISE_RTOL


@pytest.mark.parametrize('B,N,Z,h', [(4099, 15, 6, 185), (1, 15, 7, 185), (777, 5, 6, 96), (20000, 6, 7, 32), (3000, 15, 7, 128),
                                     (500, 9, 8, 190), (17, 1, 1, 14)])
def test_precise_mode_random_batches(crl, B, N, Z, h):
    """crl_zone_encode_precise against the float64 reference's per-element bound and against the fp32 module (1e-4);
    in_dim 16 (the widest the precise kernel takes), h 190, N 1."""
    gen = torch.Generator(device='cuda').manual_seed(B + h + 1)
    rn = lambda *s_, scale=1.0: (torch.randn(*s_, device='cuda', generator=gen) * scale)
    sd = {'zone_net_.0.weight': rn(h, 8 + Z, scale=0.4), 'zone_net_.0.bias': rn(h, scale=0.2),
          'zone_net_.2.weight': rn(h, h, scale=1.5 / h ** 0.5), 'zone_net_.2.bias': rn(h, scale=0.2),
          'zone_net_.4.weight': rn(h, h, scale=1.5 / h ** 0.5), 'zone_net_.4.bias': rn(h, scale=0.2),
          'combine_net_.weight': rn(h, 8 + h, scale=0.1), 'combine_net_.bias': rn(h, scale=0.1)}
    obs, zobs = rn(B, 8), rn(B, N, Z)
    enc = crl.ZoneEncoder(sd, num_zones=N)
    out = torch.full((B + 3, h), 7.0, device='cuda')
    pooled = enc.pooled_precise(obs, zobs, out=out[:B])
    emb = torch.nn.functional.linear(pooled.double(), sd['zone_net_.4.weight'].double(), sd['zone_net_.4.bias'].double()).float()
    torch.cuda.synchronize()
    assert enc.healthy() and bool((out[B:] == 7.0).all()) and bool((pooled >= 0).all())
    want = fp32_ref(sd, obs, zobs)
    err = float((emb - want).abs().max()) / max(1.0, float(want.abs().max()))
    ratio, same = ref.err_ratio(pooled, *_bound_of(sd, obs, zobs, precise=True))
    print(f'precise B={B} N={N} Z={Z} h={h}: {err:.2e} of the largest reference value, largest |err|/r {ratio:.3f}')
    assert err <= PRECISE_RTOL and same and ratio <= 1.0
