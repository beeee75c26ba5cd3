"""CPU-side checks of the product's host logic and of the kernel's per-env arithmetic
compiled for the host (tests/hostcheck): no GPU needed."""
import ctypes
import itertools
import math
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import mj_point as mj
from oracle import zone_env as ze

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HC = os.path.join(ROOT, 'tests', 'hostcheck')


@pytest.fixture(scope='module')
def hc():
    so = os.path.join(HC, 'libhostcheck.so')
    src = os.path.join(HC, 'hostcheck.cpp')
    core = os.path.join(ROOT, 'combinatorial_rl_tasks_b200', 'csrc', 'crl_core.cuh')
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(core)):
        subprocess.run(['g++', '-O2', '-x', 'c++', '-shared', '-fPIC', '-o', so, src], check=True)
    L = ctypes.CDLL(so)
    fp = ctypes.POINTER(ctypes.c_float)
    L.hc_substeps.argtypes = [fp, ctypes.c_float, ctypes.c_float, ctypes.c_int, fp]
    L.hc_wrap_pi.restype = ctypes.c_float
    L.hc_wrap_pi.argtypes = [ctypes.c_float]
    L.hc_sqrt_threshold.restype = ctypes.c_double
    L.hc_sqrt_threshold.argtypes = [ctypes.c_double]
    L.hc_inside_zone.argtypes = [ctypes.c_float] * 4 + [ctypes.c_double]
    L.hc_hamming.argtypes = [ctypes.c_uint32, ctypes.c_int]
    L.hc_philox.argtypes = [ctypes.c_void_p] * 3
    L.hc_div_const.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p]
    return L


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads without a GPU and exports all of include/crl_b200.h."""
    from combinatorial_rl_tasks_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'crl_b200.h')).read()
    declared = set(re.findall(r'\b(crl_[a-z_0-9]+)\s*\(', hdr))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.crl_abi_version() == 9
    assert not hasattr(lib, 'crl_step_host_delta')
    assert b'NULL' in lib.crl_strerror(-1)


def test_argument_errors_are_detected_on_the_host():
    from combinatorial_rl_tasks_b200 import _lib
    lib = _lib.load()
    cfg = _lib.CrlConfig(task=0, num_envs=64, num_zones=15, num_steps=2000, frameskip=10, max_cooldown=150,
                         zone_size=0.2)
    sizes = (ctypes.c_int64 * 23)()
    assert lib.crl_plane_bytes(cfg, sizes, 23) == 0
    assert list(sizes) == [1024, 1024, 7680, 0, 0, 512, 256, 1024, 64, 2 * 7680, 0, 2 * 1024, 2 * 512, 2 * 256,
                           2048, 64 * 90 * 4, 512, 24, 16 * 129, 16, 256, 256, 16]
    rd, wr = ctypes.c_int64(), ctypes.c_int64()
    assert lib.crl_step_bytes(cfg, ctypes.byref(rd), ctypes.byref(wr)) == 0 and (rd.value, wr.value) == (160, 432)
    bad = _lib.CrlConfig(task=7, num_envs=64, num_zones=15, num_steps=2000, zone_size=0.2)
    assert lib.crl_plane_bytes(bad, sizes, 23) == -2
    st, out = _lib.CrlState(), _lib.CrlOut()
    assert lib.crl_step(cfg, st, None, out, 0, 0, 0, None) == -1          # NULL planes
    cfg2 = _lib.CrlConfig(task=0, num_envs=64, num_zones=9, num_steps=2000, frameskip=10, zone_size=0.2)
    buf = (ctypes.c_char * 4096)()
    a = ctypes.addressof(buf)
    a16 = (a + 15) & ~15
    st = _lib.CrlState(pose=a16, aux=a16, zone_xy=a16, seed=a16, episode=a16, origin=a16, counters=a16)
    out = _lib.CrlOut(obs=a16, zone_obs=a16, result=a16)
    assert lib.crl_step(cfg2, st, None, out, 0, 0, 0, None) == -4         # no kernel for N = 9
    assert lib.crl_step(cfg, st, None, out, _lib.STEP_CHAINED, 0, 0, None) == -1   # chained needs CrlState.stamp
    assert lib.crl_step(cfg, st, None, out, _lib.STEP_TRACK_ROWS, 0, 0, None) == -1  # needs CrlState.row_list
    call = ctypes.c_void_p()
    assert lib.crl_host_call_create(cfg, st, out, out, 0, ctypes.byref(call)) == -1   # no row_list
    assert lib.crl_host_call_step(None, a16, None) == -1 and not call.value
    lib.crl_host_call_destroy(None)                                        # a no-op
    st.pose = a16 + 4
    assert lib.crl_step(cfg, st, None, out, 0, 0, 0, None) == -3          # misaligned plane


def test_hard_instance_specs_and_config_checks():
    """PointTSP-v4 / v5 (main/envs/__init__.py:52-81): the product's registry against the oracle's
    independent restatement of the same configs; the fixed-placement table; initial_visited is
    validated on the host."""
    from combinatorial_rl_tasks_b200 import _lib
    from combinatorial_rl_tasks_b200.config import ENV_SPECS, TaskSpec
    from oracle import zone_env as ze
    for env_id, h in ze.HARD.items():
        spec = ENV_SPECS[env_id]
        assert (spec.task, spec.num_zones, spec.num_steps) == (_lib.TASK_TSP, h['num_zones'], h['num_steps'])
        assert spec.goals == (env_id in ze.GOAL_ENV_IDS)
        assert spec.initial_visited == sum(1 << i for i, c in enumerate(h['zones_colours']) if c == 5)
        t = spec.fixed_layout()
        assert t.shape == (16, 4) and t.dtype == np.float32
        assert tuple(t[0, :2]) == tuple(np.float32(h['robot_locations'][0]))
        assert t[0, 3] == (3 if h['robot_rot'] is not None else 1)
        n = len(h['zones_locations'])
        assert np.array_equal(t[1:1 + n, :2], np.array(h['zones_locations'], dtype=np.float32))
        assert np.all(t[1:1 + n, 3] == 1) and not t[1 + n:].any()
        # the cities are exactly the zones that do not start visited
        assert spec.initial_visited == ((1 << 15) - 1) & ~((1 << n) - 1)
    assert ENV_SPECS['PointTSP-v0'].fixed_layout() is None and ENV_SPECS['PointTSP-v0'].initial_visited == 0
    with pytest.raises(ValueError):                      # two fixed zones closer than 2 x 0.55
        TaskSpec(_lib.TASK_TSP, 5, 1000, 6, zones_locations=((0, 0), (0.5, 0.5))).fixed_layout()
    lib = _lib.load()
    sizes = (ctypes.c_int64 * 22)()
    ok = _lib.CrlConfig(task=0, num_envs=64, num_zones=15, num_steps=1000, zone_size=0.2, initial_visited=0x7fe0)
    assert lib.crl_plane_bytes(ok, sizes, 22) == 0
    bad = _lib.CrlConfig(task=0, num_envs=64, num_zones=15, num_steps=1000, zone_size=0.2, initial_visited=0x8000)
    assert lib.crl_plane_bytes(bad, sizes, 23) == -2     # a bit beyond zone N - 1
    assert ctypes.sizeof(_lib.CrlConfig) == 112 and ctypes.sizeof(_lib.CrlState) == 23 * 8


def test_design_twin_honours_fixed_placements():
    """oracle/crl_oracle.c ph_reset with the fixed-placement table: fixed objects at their
    places, sampled ones inside the arena and clear of every keepout, v4's heading fixed."""
    from combinatorial_rl_tasks_b200.config import ENV_SPECS
    for env_id in ('PointTSP-v4', 'PointTSP-v5'):
        spec = ENV_SPECS[env_id]
        t = spec.fixed_layout()
        n = len(spec.zones_locations)
        rots = []
        for seed in range(40):
            tw = co.philox_reset(env_id, seed, fixed=t)
            assert np.array_equal(tw['xy0'], t[0, :2]) and np.array_equal(tw['zone_xy'][:n], t[1:1 + n, :2])
            pts = np.concatenate([tw['xy0'][None], tw['zone_xy']]).astype(np.float64)
            keep = np.array([0.4] + [0.55] * 15)
            d = np.linalg.norm(pts[:, None] - pts[None], axis=2) + 1e9 * np.eye(16)
            assert np.all(d >= keep[:, None] + keep[None] - 1e-5)
            assert np.abs(tw['zone_xy'][n:]).max() <= 2.45 + 1e-6
            rots.append(tw['rot0'])
        assert (set(rots) == {-1.0}) if spec.robot_rot is not None else (len(set(rots)) == 40)
        free = co.philox_reset(env_id, 3)                # same seed, nothing fixed: a different map
        assert not np.array_equal(free['xy0'], t[0, :2])


def test_integration_md_structs_match_the_binding():
    """The ctypes structs printed in INTEGRATION.md section 2 (executed as written by a GPU test) declare the
    same fields, in the same order and of the same size, as the product's own binding and the C header."""
    from combinatorial_rl_tasks_b200 import _lib
    md = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    sec = md[md.index('## 2. Bind the C ABI directly'):]
    code = re.search(r'```python\n(.*?)```', sec, re.S).group(1)
    defs = code[code.index('class CrlConfig'):code.index('cfg = CrlConfig')]
    ns = {'ctypes': ctypes}
    exec(defs, ns)
    for name in ('CrlConfig', 'CrlState', 'CrlOut'):
        mine, theirs = getattr(_lib, name), ns[name]
        assert [f[0] for f in mine._fields_] == [f[0] for f in theirs._fields_], name
        assert ctypes.sizeof(mine) == ctypes.sizeof(theirs), name
    hdr = open(os.path.join(ROOT, 'include', 'crl_b200.h')).read()
    body = hdr[hdr.index('typedef struct CrlState {'):hdr.index('} CrlState;')]
    fields = re.findall(r'\b(\w+);', re.sub(r'/\*.*?\*/', '', body, flags=re.S))
    assert fields == [f[0] for f in _lib.CrlState._fields_]


def test_encoder_shape_checks_run_on_the_host():
    """crl_encoder_packed_bytes: limits of the tcgen05 zone encoder are refused before anything is launched."""
    from combinatorial_rl_tasks_b200 import _lib
    lib = _lib.load()
    n = ctypes.c_int64()
    S = _lib.CrlEncoderShape
    assert lib.crl_encoder_packed_bytes(S(8, 6, 185, 15), ctypes.byref(n)) == 0 and n.value == 256 * 192 * 2 + 256 * 32
    assert lib.crl_encoder_packed_bytes(S(8, 7, 64, 6), ctypes.byref(n)) == 0 and n.value == 128 * 80 * 2 + 128 * 32
    assert lib.crl_encoder_packed_bytes(S(8, 6, 190, 15), ctypes.byref(n)) == 0
    assert lib.crl_encoder_packed_bytes(S(8, 6, 191, 15), ctypes.byref(n)) == -4     # W2 + operand buffers exceed an SM
    assert lib.crl_encoder_packed_bytes(S(10, 7, 185, 15), ctypes.byref(n)) == 0 and n.value == 256 * 192 * 2 + 256 * 64   # 32-wide input
    assert lib.crl_encoder_packed_bytes(S(20, 12, 64, 15), ctypes.byref(n)) == -2    # no room for the ones column
    assert lib.crl_encoder_packed_bytes(S(8, 6, 64, 17), ctypes.byref(n)) == -2      # more than 16 zone slots
    assert lib.crl_encoder_packed_bytes(None, ctypes.byref(n)) == -1
    assert lib.crl_zone_encode(S(8, 6, 185, 15), 64, None, None, None, None, None, None) == -1


def test_encoder_fails_loudly_without_cuda():
    torch = pytest.importorskip('torch')
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    import combinatorial_rl_tasks_b200 as crl
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        crl.ZoneEncoder({}, num_zones=15)


def test_vec_env_fails_loudly_without_cuda():
    torch = pytest.importorskip('torch')
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    import combinatorial_rl_tasks_b200 as crl
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        crl.ZoneVecEnv('PointTSP-v0', 8)


def test_philox_known_answers(hc):
    """Random123 kat_vectors, philox4x32-10."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        c, k, o = np.array(ctr, np.uint32), np.array(key, np.uint32), np.zeros(4, np.uint32)
        hc.hc_philox(c.ctypes.data, k.ctypes.data, o.ctypes.data)
        assert tuple(o) == want
        co.lib().ph_philox(c.ctypes.data, k.ctypes.data, o.ctypes.data)     # the oracle's twin agrees
        assert tuple(o) == want


def test_zone_predicate_is_numpy_exact(hc):
    t2 = hc.hc_sqrt_threshold(0.2)
    assert math.sqrt(t2) <= 0.2 < math.sqrt(np.nextafter(t2, 1.0))
    rs = np.random.RandomState(0)
    n_in = 0
    for k in range(60000):
        z = rs.uniform(-2.5, 2.5, 2).astype(np.float32)
        ang, r = rs.uniform(0, 2 * np.pi), 0.2 + rs.choice([0.0, 1e-9, -1e-9, 3e-8, -3e-8, 1e-6, -1e-6, 0.05, -0.05])
        p = (z.astype(np.float64) + r * np.array([math.cos(ang), math.sin(ang)])).astype(np.float32)
        ref = bool(np.sqrt(np.sum(np.square(z.astype(np.float64) - p.astype(np.float64)))) <= 0.2)
        got = bool(hc.hc_inside_zone(float(p[0]), float(p[1]), float(z[0]), float(z[1]), t2))
        assert got == ref, (k, z, p)
        n_in += ref
    assert 6000 < n_in < 54000


def test_hamming_exhaustive(hc):
    for cols in itertools.product(range(3), repeat=6):
        word = sum(c << (2 * i) for i, c in enumerate(cols))
        assert hc.hc_hamming(word, 6) == ze.hamming_to_goal(np.array(cols))


def test_constant_division_equals_the_reference_values(hc):
    """The kernel divides small integers by num_steps / max_cooldown with a reciprocal multiply and
    one exact-remainder correction.  It must equal what the reference computes in fp64 and the
    consumer casts to float32 (format.py:27-28): zone time (zone_max_steps - steps) / max_steps
    (TTSP_env.py:25), remaining 1 - steps / num_steps (ZoneEnvBase.py:190-192), and
    np.float32(cooldown) / 150 (colour_match_env.py:79)."""
    for d in (2000, 1000, 300, 150, 7, 1999, 65535):
        lo, hi = -65535, 65535
        out = np.zeros(hi - lo + 1, dtype=np.float32)
        assert hc.hc_div_const(d, lo, hi, out.ctypes.data) == 1, d
        n = np.arange(lo, hi + 1, dtype=np.float64)
        assert np.array_equal(out, (n / d).astype(np.float32)), d
        assert np.array_equal(out, np.arange(lo, hi + 1).astype(np.float32) / np.float32(d)), d
    steps = np.arange(0, 2001, dtype=np.float64)
    out = np.zeros(2001, dtype=np.float32)
    hc.hc_div_const(2000, 0, 2000, out.ctypes.data)
    assert np.array_equal(out[::-1], (1.0 - steps / 2000).astype(np.float32))
    out = np.zeros(256, dtype=np.float32)
    hc.hc_div_const(150, 0, 255, out.ctypes.data)
    assert np.array_equal(out, (np.arange(256).astype(np.float32) / 150).astype(np.float64).astype(np.float32))


def test_closed_form_substep_vs_oracle(hc):
    """The kernel's closed-form (M + hB)^-1 solve, compiled for the host, against the
    oracle's generic 3x3 solve: 1e-5 relative per substep from identical inputs."""
    rs = np.random.RandomState(0)
    fp = ctypes.POINTER(ctypes.c_float)
    cs = (ctypes.c_float * 2)()
    worst = 0.0
    for trial in range(2000):
        st = np.array([rs.uniform(-2.5, 2.5), rs.uniform(-2.5, 2.5), rs.uniform(-np.pi, np.pi),
                       rs.uniform(-1.5, 1.5), rs.uniform(-1.5, 1.5), rs.uniform(-4.5, 4.5)], dtype=np.float32)
        a = rs.uniform(-1.3, 1.3, 2).astype(np.float32)
        if trial % 3 == 0:
            a[0] *= 0.04
        if trial % 5 == 0:
            a[1] = np.float32(0.3 * st[5] + rs.uniform(-0.04, 0.04))
        w = st.astype(np.float64)
        q_ref, v_ref = mj.substep(w[:3], w[3:], a.astype(np.float64))     # rot0 = 0: world == qpos frame
        out = st.copy()
        hc.hc_substeps(out.ctypes.data_as(fp), float(a[0]), float(a[1]), 1, cs)
        ref = np.concatenate([q_ref, v_ref])
        err = np.abs(out - ref) / np.maximum(1.0, np.abs(ref))
        worst = max(worst, err.max())
        assert abs(cs[0] - math.cos(q_ref[2])) < 2e-6 and abs(cs[1] - math.sin(q_ref[2])) < 2e-6
    assert worst <= 1e-5, worst


def test_wrap_pi(hc):
    for x in np.linspace(-3.3, 3.3, 1001):
        y = hc.hc_wrap_pi(float(x))
        assert -math.pi - 1e-6 <= y <= math.pi + 1e-6
        assert abs(math.remainder(y - x, 2 * math.pi)) < 5e-7


def test_philox_reset_twin_layouts_are_valid():
    """The design twin of the device reset: keepouts, extents, Beta(3,1.5) timeouts."""
    tm_all = []
    for seed in range(200):
        r = co.philox_reset('PointTTSP-v0', seed)
        pts = np.vstack([r['xy0'][None], r['zone_xy']]).astype(np.float64)
        keep = np.array([0.4] + [0.55] * 15)
        assert np.all(np.abs(pts) <= 3.0 - keep[:, None] + 1e-6)
        d = np.linalg.norm(pts[:, None] - pts[None], axis=2)
        need = keep[:, None] + keep[None]
        iu = np.triu_indices(16, 1)
        assert np.all(d[iu] >= need[iu] - 1e-6)
        assert 0.0 <= r['rot0'] < 2 * np.pi + 1e-6 and r['seed_after'] == seed + 1
        tm_all.append(r['zone_max_steps'])
    tm = np.concatenate(tm_all) / 2000.0
    # Beta(3, 1.5): mean 2/3, variance ab/((a+b)^2 (a+b+1)) = 0.0404
    assert abs(tm.mean() - 2 / 3) < 0.015 and abs(tm.var() - 0.0404) < 0.004
    cols = np.concatenate([co.philox_reset('ColourMatch-v0', s)['colours'] for s in range(2000)])
    assert np.all(np.abs(np.bincount(cols, minlength=3) / len(cols) - 1 / 3) < 0.02)


def test_timeout_wrapper_matches_the_reference_class():
    """compat.TimeoutWrapper against the REAL main/envs/wrappers.py:161-194 on a scripted inner env: the reference class's
    trace (imported over the gym / mujoco_py / glfw stubs of tests/golden/stubs, which it matched when compat.TimeoutWrapper
    was written) is stored in tests/golden/timeout_wrapper_trace.json, as JSON (tuples read back as lists)."""
    import json
    from combinatorial_rl_tasks_b200.compat import TimeoutWrapper

    class Inner:
        observation_space = action_space = None

        def __init__(self):
            self.t = 0

        def reset(self):
            self.t = 0
            return ('obs', 0)

        def step(self, action):
            self.t += 1
            return ('obs', self.t), 1.5 * self.t, self.t == 4, {'inner': True}

    def trace(w):
        out = [w.reset()]
        for k in range(9):
            out.append(w.step(k))
        out.append(w.reset())
        out.append(w.step(0))
        return out

    ours = trace(TimeoutWrapper(Inner(), max_timeout=7))
    # steps 1-3 pass through, step 4 ends the inner env (reward kept, done hidden), 5-6 repeat its last obs with reward
    # 0, step 7 raises done; the timer keeps counting past max_timeout without raising done again
    assert ours[1] == (('obs', 1), 1.5, False, {'timer': 1}) and ours[4] == (('obs', 4), 6.0, False, {'timer': 4})
    assert ours[5] == (('obs', 4), 0, False, {'timer': 5}) and ours[7] == (('obs', 4), 0, True, {'timer': 7})
    assert ours[8] == (('obs', 4), 0, False, {'timer': 8}) and ours[10] == ('obs', 0) and ours[11][3] == {'timer': 1}
    with open(os.path.join(ROOT, 'tests', 'golden', 'timeout_wrapper_trace.json')) as f:
        real = json.load(f)
    assert len(real) == len(ours) == 12
    assert json.loads(json.dumps(ours)) == real
