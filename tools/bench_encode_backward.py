"""Forward + backward of ZoneEnvModel's (B N)-row part -- pooled = mean_z relu(W2 relu(W1 x + b1) + b2) and the
gradients of W1, b1, W2, b2 for a given dL/dpooled -- three ways, timed with CUDA events:

  fused     FusedZoneEnvModel.pooled + backward: crl_encoder_pack, crl_zone_encode, crl_zone_encode_backward (+ its
            fixed-order reduction), i.e. everything a training step pays for this part
  fp32      torch eager, fp32 (what the reference's update runs)
  bf16      torch eager under autocast(bfloat16)

Cases: PointTSP (N 15, Z 6) h = 185 at 65,536 envs, ColourMatch (N 6, Z 7) h = 64 at 262,144 envs.  Each case cycles
through enough input sets (obs, zone_obs, g) to exceed the 126 MB L2, warms up every path first, and reports the
median of the timed iterations.  TFLOP/s use the algorithmic count of forward + backward (no input gradients):
B N (6 h^2 + 4 h in_dim) -- the fused path's recomputed forward is not counted -- against the 2,250 TFLOP/s dense bf16
data-sheet figure.  Prints one JSON line.

    python tools/bench_encode_backward.py [--iters 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import combinatorial_rl_tasks_b200 as crl  # noqa: E402

PEAK_BF16 = 2250e12
L2_BYTES = 126 * 2 ** 20
CASES = [('PointTSP', 65536, 15, 6, 185), ('ColourMatch', 262144, 6, 7, 64)]


def flops(B, N, in_dim, h):
    return B * N * (6 * h * h + 4 * h * in_dim)


def torch_zone(l1, l2, obs, zobs):
    x = torch.cat([obs[:, None, :].expand(-1, zobs.shape[1], -1), zobs], -1)
    return torch.relu(l2(torch.relu(l1(x)))).mean(1)


def time_it(fn, sets, iters, warmup):
    for i in range(warmup):
        fn(*sets[i % len(sets)])
    torch.cuda.synchronize()
    ts = []
    for i in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(*sets[i % len(sets)])
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device (sm_100a)')
    torch.backends.cuda.matmul.allow_tf32 = False
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True).stdout.strip()
    res = {'device': torch.cuda.get_device_name(0), 'nvidia_smi': q, 'iters': args.iters, 'cases': []}
    for name, B, N, Z, h in CASES:
        in_dim = 8 + Z
        gen = torch.Generator(device='cuda').manual_seed(0)
        model = crl.FusedZoneEnvModel(8, Z, N, h)
        l1, l2 = model.zone_net_[0], model.zone_net_[2]
        per_set = 4 * B * (8 + N * Z + h)
        n_sets = max(2, -(-2 * L2_BYTES // per_set))
        sets = [(torch.randn(B, 8, device='cuda', generator=gen), torch.rand(B, N, Z, device='cuda', generator=gen),
                 torch.randn(B, h, device='cuda', generator=gen) * 1e-3) for _ in range(n_sets)]

        def fused(o, z, g):
            l1.weight.grad = None
            model.pooled(o, z).backward(g)

        def eager(o, z, g):
            l1.weight.grad = None
            torch_zone(l1, l2, o, z).backward(g)

        def autocast(o, z, g):
            l1.weight.grad = None
            with torch.autocast('cuda', dtype=torch.bfloat16):
                p = torch_zone(l1, l2, o, z)
            p.float().backward(g)

        t = {k: time_it(fn, sets, args.iters, args.warmup) for k, fn in (('fused', fused), ('fp32', eager), ('bf16_autocast', autocast))}
        f = flops(B, N, in_dim, h)
        res['cases'].append({'case': name, 'B': B, 'N': N, 'in_dim': in_dim, 'h': h, 'input_sets': n_sets,
                             'gflop': f / 1e9, 'ms': {k: v * 1e3 for k, v in t.items()},
                             'tflops': {k: f / v / 1e12 for k, v in t.items()},
                             'share_of_bf16_peak': {k: f / v / PEAK_BF16 for k, v in t.items()},
                             'fused_speedup': {'vs_fp32': t['fp32'] / t['fused'], 'vs_bf16_autocast': t['bf16_autocast'] / t['fused']},
                             'healthy': model.healthy()})
        del sets, model
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == '__main__':
    main()
