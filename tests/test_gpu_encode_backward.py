"""crl_zone_encode_backward (tcgen05, csrc/crl_encode.cu) and FusedZoneEnvModel, the trainable ZoneEnvModel built on it.

* Every element of dW1, db1, dW2, db2 against the float64 reference's per-element bound
  (tests/_encoder_backward_reference.py) over the forward test's shape classes and the backward's own tile edges; inputs
  and g are views with NaN past row B, outputs have guard elements.  The largest |err| / r per shape is printed.
* Two calls give bit-identical results (fixed-order fp64 reduction of per-CTA partials, no atomics).
* NaN in g or in an input row: non-finite exactly where the reference is.
* FusedZoneEnvModel against torch fp32 autograd on the same weights (relative Frobenius error per parameter gradient),
  its guards, and examples/collect_ppo.py --fused-train.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from tests import _encoder_backward_reference as bref  # noqa: E402
from tests import _encoder_reference as ref  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'model_zone_env.npz')
# Relative Frobenius error of a parameter gradient against torch fp32 autograd.  With bf16 operands the gradients of the
# first two Linears are dominated by relu masks that the rounding flips (a flipped mask moves a whole term), so under a
# zero-mean random loss the error is about sqrt(fraction of flipped masks): 1.4-2.7e-2 for the golden weights, the same
# for torch's own bf16 autocast training of the module (a float32 emulation of the kernel's algorithm gives the same
# figures).  ZONE_RTOL is the stated bar for those four gradients; on top of it the fused gradients must be no further
# from fp32 than AUTOCAST_FACTOR times what bf16 autocast gets.  The B-row head's gradients see only bf16 `pooled`.
ZONE_RTOL = 5e-2
AUTOCAST_FACTOR = 1.25
HEAD_RTOL = 1e-2


@pytest.fixture(scope='module')
def crl():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    import combinatorial_rl_tasks_b200 as m
    return m


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _weights(gen, h, in_dim, D):
    rn = lambda *s, scale=1.0: (torch.randn(*s, device='cuda', generator=gen) * scale)
    return {'zone_net_.0.weight': rn(h, in_dim, scale=0.4), 'zone_net_.0.bias': rn(h, scale=0.2),
            'zone_net_.2.weight': rn(h, h, scale=1.5 / h ** 0.5), 'zone_net_.2.bias': rn(h, scale=0.2)}


def _nan_tail(t):
    buf = torch.full((t.shape[0] + 40,) + tuple(t.shape[1:]), float('nan'), device=t.device)
    buf[:t.shape[0]] = t
    return buf[:t.shape[0]]


def _backward(sd, N, obs, zobs, g):
    """The C ABI directly: pack, workspace, backward; outputs with guard elements of 7.0 on both sides."""
    from combinatorial_rl_tasks_b200 import _lib
    lib = _lib.load()
    w1, b1, w2, b2 = (sd[f'zone_net_.{k}'] for k in ('0.weight', '0.bias', '2.weight', '2.bias'))
    h, in_dim = w1.shape
    B, D = obs.shape
    shape = _lib.CrlEncoderShape(D, in_dim - D, h, N)
    s0 = torch.cuda.current_stream().cuda_stream
    n = ctypes.c_int64()
    _lib.check(lib.crl_encoder_packed_bytes(shape, ctypes.byref(n)))
    packed = torch.zeros(n.value, dtype=torch.uint8, device='cuda')
    _lib.check(lib.crl_encoder_pack(shape, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), packed.data_ptr(), s0))
    _lib.check(lib.crl_encoder_backward_workspace_bytes(shape, B, ctypes.byref(n)))
    ws = torch.empty(n.value, dtype=torch.uint8, device='cuda')
    sizes = {'dw1': (h, in_dim), 'db1': (h,), 'dw2': (h, h), 'db2': (h,)}
    bufs = {k: torch.full((int(np.prod(s)) + 8,), 7.0, device='cuda') for k, s in sizes.items()}
    outs = {k: bufs[k][4:-4].view(sizes[k]) for k in sizes}
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    _lib.check(lib.crl_zone_encode_backward(shape, B, obs.data_ptr(), zobs.data_ptr(), packed.data_ptr(), g.data_ptr(),
                                            ws.data_ptr(), outs['dw1'].data_ptr(), outs['db1'].data_ptr(),
                                            outs['dw2'].data_ptr(), outs['db2'].data_ptr(), status.data_ptr(), s0))
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    for k, b in bufs.items():
        assert bool((b[:4] == 7.0).all()) and bool((b[-4:] == 7.0).all()), k
    return outs


def _bound(sd, obs, zobs, g):
    return bref.backward_bound(sd['zone_net_.0.weight'], sd['zone_net_.0.bias'], sd['zone_net_.2.weight'],
                               sd['zone_net_.2.bias'], obs, zobs, g, _sms())


# (B, N, Z, h, D): the forward test's shapes (N 1..16, both slot counts; h 1..190; in_dim 2..31, one and two K steps;
# B 1 and the forward's tile edges, 65,536) plus PointTSP's own shape at 65,536 envs and the backward's tile edges (4
# envs per tile for 16 slots, 8 for 8: B 3, 4, 5, 7, 8, 9, 15, 16, 17)
SHAPES = [(4099, 15, 6, 185, 8), (1, 15, 7, 185, 8), (777, 5, 6, 96, 8), (20000, 6, 7, 32, 8), (3001, 15, 7, 185, 10),
          (515, 6, 7, 64, 16),
          (1, 1, 1, 1, 1), (15, 5, 7, 14, 8), (16, 7, 8, 31, 8), (17, 8, 6, 126, 8), (7, 9, 6, 129, 24),
          (8, 16, 15, 160, 16), (9, 15, 6, 189, 8), (91, 16, 7, 189, 1), (3001, 5, 14, 190, 1), (515, 7, 7, 160, 24),
          (1000, 1, 22, 129, 8), (65536, 8, 6, 126, 8),
          (65536, 15, 6, 185, 8), (3, 15, 6, 185, 8), (4, 16, 7, 64, 8), (5, 12, 7, 100, 8)]


@pytest.mark.parametrize('B,N,Z,h,D', SHAPES)
def test_gradients_inside_the_bound(crl, B, N, Z, h, D):
    gen = torch.Generator(device='cuda').manual_seed(B + h + 7)
    sd = _weights(gen, h, D + Z, D)
    obs = _nan_tail(torch.randn(B, D, device='cuda', generator=gen))
    zobs = _nan_tail(torch.randn(B, N, Z, device='cuda', generator=gen))
    g = _nan_tail(torch.randn(B, h, device='cuda', generator=gen))
    out = _backward(sd, N, obs, zobs, g)
    want = _bound(sd, obs, zobs, g)
    ratios = {}
    for k, (c, r) in want.items():
        ratio, same = ref.err_ratio(out[k], c, r)
        ratios[k] = ratio
        assert same, (k, 'non-finite where the reference is finite, or the reverse')
        assert ratio <= 1.0, (k, ratio)
    print(f'B={B} N={N} Z={Z} h={h} D={D}: largest |err|/r ' + ', '.join(f'{k} {v:.3f}' for k, v in ratios.items()))
    again = _backward(sd, N, obs, zobs, g)
    for k in out:
        assert torch.equal(out[k], again[k]), k                  # bit-identical from run to run


@pytest.mark.parametrize('where', ['g', 'input'])
def test_non_finite_inputs(crl, where):
    """A NaN in g (two elements) or in one input row (a zone row, an obs row): the outputs are non-finite exactly where
    the float64 reference is, and inside the bound elsewhere."""
    B, N, Z, h = 3001, 15, 6, 185
    gen = torch.Generator(device='cuda').manual_seed(23)
    sd = _weights(gen, h, 8 + Z, 8)
    obs = torch.randn(B, 8, device='cuda', generator=gen)
    zobs = torch.randn(B, N, Z, device='cuda', generator=gen)
    g = torch.randn(B, h, device='cuda', generator=gen)
    if where == 'g':
        g[17, 5] = float('nan')
        g[B - 1, 100] = float('nan')
    else:
        zobs[40, 3, 2] = float('nan')
        obs[B - 1, 6] = float('nan')
    out = _backward(sd, N, obs, zobs, g)
    want = _bound(sd, obs, zobs, g)
    ratios = {}
    for k, (c, r) in want.items():
        ratio, same = ref.err_ratio(out[k], c, r)
        ratios[k] = ratio
        if k == 'dw2':
            assert not bool(torch.isfinite(c).all())             # the NaN reaches the outputs
        assert same, (k, int((~torch.isfinite(out[k])).sum()), int((~torch.isfinite(c)).sum()))
        assert ratio <= 1.0, (k, ratio)
    print(f'NaN in {where}: largest |err|/r over the finite elements ' + ', '.join(f'{k} {v:.3f}' for k, v in ratios.items()))


def _golden(tag):
    g = dict(np.load(GOLDEN))
    sd = {k[len(tag) + 4:]: torch.from_numpy(g[k]).cuda() for k in g if k.startswith(tag + '_sd_')}
    return sd, torch.from_numpy(g[f'{tag}_obs']).cuda(), torch.from_numpy(g[f'{tag}_zone_obs']).cuda(), g[f'{tag}_out']


class _TorchZoneEnvModel(torch.nn.Module):
    """The reference's ZoneEnvModel (env_model.py:48-79) in plain torch fp32."""

    def __init__(self, obs_dim, zone_dim, h):
        super().__init__()
        self.zone_net_ = torch.nn.Sequential(torch.nn.Linear(obs_dim + zone_dim, h), torch.nn.ReLU(), torch.nn.Linear(h, h),
                                             torch.nn.ReLU(), torch.nn.Linear(h, h))
        self.combine_net_ = torch.nn.Linear(obs_dim + h, h)

    def forward(self, obs):
        o, z = obs['obs'], obs['zone_obs']
        x = torch.cat([o[:, None, :].expand(-1, z.shape[1], -1), z], -1)
        return self.combine_net_(torch.cat([o, self.zone_net_(x).sum(1) / z.shape[1]], -1))


@pytest.mark.parametrize('tag,n', [('tsp', 15), ('cm', 6)])
def test_autograd_against_torch_fp32(crl, tag, n):
    """FusedZoneEnvModel loads the golden ZoneEnvModel weights strictly, its forward matches the recorded fp32 output,
    and for a scalar loss on a 4,096-env batch every parameter gradient agrees with torch fp32 autograd on the same
    module (relative Frobenius error; the B-row head's too), at most as far from it as torch bf16 autocast's."""
    sd, obs, zobs, out_ref = _golden(tag)
    h, in_dim = sd['zone_net_.0.weight'].shape
    model = crl.FusedZoneEnvModel(8, in_dim - 8, n, h)
    model.load_state_dict(sd, strict=True)
    assert set(model.state_dict()) == set(sd)
    twin = _TorchZoneEnvModel(8, in_dim - 8, h).cuda()
    twin.load_state_dict(sd, strict=True)
    torch.backends.cuda.matmul.allow_tf32 = False
    # the forward: pooled inside the forward's bound, the output within 1e-2 of the recorded fp32 module's
    with torch.no_grad():
        pooled = model.pooled(obs, zobs)
        y = model({'obs': obs, 'zone_obs': zobs}).cpu().numpy()
    ratio, same = ref.err_ratio(pooled, *ref.pooled_bound(sd['zone_net_.0.weight'], sd['zone_net_.0.bias'],
                                                          sd['zone_net_.2.weight'], sd['zone_net_.2.bias'], obs, zobs))
    e_out = float(np.abs(y - out_ref).max()) / max(1.0, float(np.abs(out_ref).max()))
    assert same and ratio <= 1.0 and e_out <= 1e-2, (ratio, e_out)
    # gradients on a bigger batch with a fixed random loss
    gen = torch.Generator(device='cuda').manual_seed(3)
    B = 4096
    o = torch.randn(B, 8, device='cuda', generator=gen)
    z = torch.rand(B, n, in_dim - 8, device='cuda', generator=gen)
    wl = torch.randn(B, h, device='cuda', generator=gen)
    auto = _TorchZoneEnvModel(8, in_dim - 8, h).cuda()
    auto.load_state_dict(sd, strict=True)
    for m in (model, twin, auto):
        m.zero_grad()
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=m is auto):
            y = m({'obs': o, 'zone_obs': z})
        (y.float() * wl).sum().backward()
    errs, errs_auto = {}, {}
    for name, p in twin.named_parameters():
        rel = lambda m: float((dict(m.named_parameters())[name].grad - p.grad).norm() / p.grad.norm())
        errs[name], errs_auto[name] = rel(model), rel(auto)
    print(f'{tag}: forward |err|/r {ratio:.3f}, out {e_out:.2e}; gradient relative Frobenius error against fp32, fused '
          '(bf16 autocast): ' + ', '.join(f'{k} {v:.2e} ({errs_auto[k]:.2e})' for k, v in errs.items()))
    for name, v in errs.items():
        if name.startswith('zone_net_.0') or name.startswith('zone_net_.2'):
            assert v <= ZONE_RTOL and v <= AUTOCAST_FACTOR * errs_auto[name] + 1e-3, (name, v, errs_auto[name])
        else:
            assert v <= HEAD_RTOL, (name, v)
    assert model.healthy()


def test_guards(crl):
    from combinatorial_rl_tasks_b200 import _lib
    sd, obs, zobs, _ = _golden('tsp')
    model = crl.FusedZoneEnvModel(8, 6, 15, 185)
    model.load_state_dict(sd)
    # an in-place optimiser step between forward and backward
    out = model({'obs': obs, 'zone_obs': zobs}).sum()
    with torch.no_grad():
        model.zone_net_[2].weight.mul_(0.5)
    with pytest.raises(RuntimeError):
        out.backward()
    # input gradients are not computed
    with pytest.raises(RuntimeError, match='obs'):
        model({'obs': obs.clone().requires_grad_(), 'zone_obs': zobs})
    # unsupported shapes: refused as the forward refuses them
    with pytest.raises(RuntimeError):
        crl.FusedZoneEnvModel(8, 6, 15, 191)
    lib = _lib.load()
    S = _lib.CrlEncoderShape
    n = ctypes.c_int64()
    assert lib.crl_encoder_backward_workspace_bytes(S(8, 6, 185, 15), 65536, ctypes.byref(n)) == 0
    assert n.value == min(16384, _sms()) * (185 + 1 + 14 + 1) * 185 * 4
    assert lib.crl_encoder_backward_workspace_bytes(S(8, 6, 191, 15), 10, ctypes.byref(n)) == -4
    assert lib.crl_encoder_backward_workspace_bytes(S(24, 8, 64, 15), 10, ctypes.byref(n)) == -2
    assert lib.crl_encoder_backward_workspace_bytes(S(8, 6, 185, 17), 10, ctypes.byref(n)) == -2
    assert lib.crl_encoder_backward_workspace_bytes(S(8, 6, 185, 15), 0, ctypes.byref(n)) == -2
    p = torch.zeros(1 << 20, dtype=torch.uint8, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    ptr, st, s0 = p.data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream
    shape = S(8, 6, 185, 15)
    assert lib.crl_zone_encode_backward(shape, 0, *[ptr] * 9, st, s0) == -2
    assert lib.crl_zone_encode_backward(shape, 4, *[ptr] * 4, None, *[ptr] * 4, st, s0) == -1
    assert lib.crl_zone_encode_backward(shape, 4, ptr, ptr, ptr + 4, *[ptr] * 6, st, s0) == -3
    assert lib.crl_zone_encode_backward(S(8, 6, 191, 15), 4, *[ptr] * 9, st, s0) == -4
    torch.cuda.synchronize()
    assert int(status.item()) == 0


def test_collect_ppo_fused_train(crl):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'examples', 'collect_ppo.py'), '--fused-train', '--envs', '2048',
                        '--frames', '16', '--updates', '2'], capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stderr
    losses = [float(line.split('loss ')[1].split(',')[0]) for line in r.stdout.splitlines() if 'loss ' in line]
    assert len(losses) == 2 and all(np.isfinite(losses)), r.stdout
