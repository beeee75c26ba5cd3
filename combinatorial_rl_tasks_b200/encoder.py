"""ZoneEncoder: the reference's ``ZoneEnvModel`` (main/src/env_model.py:48-79) for the rollout-time
forward, with the wide part of its per-zone network and the mean-pool fused into one tensor-core kernel
(include/crl_b200.h: crl_zone_encode; csrc/crl_encode.cu).  The last Linear of ``zone_net_`` is affine, so
the mean over zones is taken before it: the kernel returns ``pooled = mean_z relu(L2(relu(L1(.))))``; the rest
of the forward, ``combine_net_([obs, L3(pooled)])``, is one affine map of ``[obs, pooled]`` and runs as a second
tensor-core kernel of the same library (crl_encoder_head).  No library GEMM is called.  ``enc(obs, zone_obs)`` /
``enc.forward_from_state(env)`` run both through crl_encoder_forward: the first kernel writes the second one's bf16
operand image directly (no fp32 ``pooled`` in between), the second fetches it with one bulk copy per 128 envs.

    model = ZoneEnvModel(obs_space, h_dim)                  # the reference's module, trained as usual
    enc = ZoneEncoder(model.state_dict(), num_zones=15)     # packs zone_net_ once (repack after an update)
    emb = enc(env.obs, env.zone_obs)                        # == model(DictList(obs=..., zone_obs=...))

All GEMMs run with bf16 operands and fp32 accumulation (the reference: fp32; biases ride in the GEMMs as bf16
hi + lo pairs).  ``ZoneEncoder`` is inference only -- no autograd graph is built.  There is no CPU path: the
constructors raise without CUDA.

Training: ``FusedZoneEnvModel`` is a drop-in ``nn.Module`` for the reference's ``ZoneEnvModel`` (same parameter names,
so ``state_dict`` loads strictly either way) whose ``pooled`` runs forward AND backward on the tensor cores
(crl_zone_encode / crl_zone_encode_backward: H1 and the layer-2 pre-activation are recomputed per tile, the (B N, h)
activations and their gradients never reach memory, dW1 / db1 / dW2 / db2 are summed per CTA and reduced in a fixed
order in fp64).  The B-row rest -- ``zone_net_[4]`` and ``combine_net_`` -- is ordinary fp32 torch autograd on
``pooled``.  Gradients reach the first two Linears only; ``obs`` / ``zone_obs`` that require grad are refused.

    model = FusedZoneEnvModel(obs_dim=8, zone_dim=6, num_zones=15, hidden=185).cuda()
    model.load_state_dict(reference_model.state_dict())     # strict: the reference's keys
    loss = f(model(obs_dict)); loss.backward(); opt.step()

Both take the observations of a ``Rollout(store='frames')`` too -- ``{'obs', 'zone_frames'}``, or a minibatch gathered
from them: the kernels then build each row from its 16-byte frame record and the rollout's layout table
(crl_zone_encode_frames / crl_zone_encode_backward_frames), with the same results as on the materialised rows.
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib


class ZoneEncoder:
    def __init__(self, state_dict, num_zones, device='cuda:0'):
        if not torch.cuda.is_available():
            raise RuntimeError('ZoneEncoder needs a CUDA device (sm_100a); there is no CPU fallback')
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.num_zones = int(num_zones)
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._ws = {}
        self.load_state_dict(state_dict)

    def load_state_dict(self, state_dict):
        """(Re)pack the weights of ``zone_net_`` / keep ``combine_net_`` (after every optimiser update)."""
        f = lambda k: state_dict[k].detach().to(self.device, torch.float32).contiguous()
        w1, b1 = f('zone_net_.0.weight'), f('zone_net_.0.bias')
        w2, b2 = f('zone_net_.2.weight'), f('zone_net_.2.bias')
        self.w3, self.b3 = f('zone_net_.4.weight'), f('zone_net_.4.bias')
        self.combine_w, self.combine_b = f('combine_net_.weight'), f('combine_net_.bias')
        self.hidden = h = w1.shape[0]
        self.obs_dim = self.combine_w.shape[1] - h
        self.zone_dim = w1.shape[1] - self.obs_dim
        assert w2.shape == self.w3.shape == (h, h) and self.zone_dim > 0
        # forward() = combine_net_([obs, W3 pooled + b3]) is ONE affine map of [obs, pooled]: fold W3 into it
        wc = self.combine_w.double()
        self.fold_w = torch.cat([wc[:, :self.obs_dim], wc[:, self.obs_dim:] @ self.w3.double()], dim=1).float().contiguous()
        self.fold_b = (wc[:, self.obs_dim:] @ self.b3.double() + self.combine_b.double()).float().contiguous()
        self.shape = _lib.CrlEncoderShape(obs_dim=self.obs_dim, zone_dim=self.zone_dim, hidden=h,
                                          num_zones=self.num_zones)
        n = ctypes.c_int64()
        _lib.check(self.lib.crl_encoder_packed_bytes(self.shape, ctypes.byref(n)))
        self.packed = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_encoder_pack(self.shape, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                                 self.packed.data_ptr(), self._stream()))
        # the two heads: forward() = fold_w [obs, pooled] + fold_b, zone_embedding() = [0 | W3] [obs, pooled] + b3
        l3_w = torch.cat([torch.zeros(h, self.obs_dim, device=self.device), self.w3], dim=1).contiguous()
        _lib.check(self.lib.crl_encoder_head_packed_bytes(self.shape, ctypes.byref(n)))
        self.packed_head = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
        self.packed_l3 = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_encoder_pack_head(self.shape, self.fold_w.data_ptr(), self.fold_b.data_ptr(),
                                                      self.packed_head.data_ptr(), self._stream()))
            _lib.check(self.lib.crl_encoder_pack_head(self.shape, l3_w.data_ptr(), self.b3.data_ptr(),
                                                      self.packed_l3.data_ptr(), self._stream()))
        self._keep = (w1, b1, w2, b2, l3_w)         # alive until the pack kernels have run
        self._packed_precise = None                 # packed on first use (pooled_precise)
        self._precise_heads = {}

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def pooled(self, obs, zone_obs, out=None):
        """mean_z relu(L2(relu(L1([obs, zone_obs[:, z]])))): (B, obs_dim) f32, (B, N, Z) f32 -> (B, h) f32
        (the fused kernel)."""
        B = obs.shape[0]
        assert obs.shape == (B, self.obs_dim) and zone_obs.shape == (B, self.num_zones, self.zone_dim)
        assert obs.dtype == zone_obs.dtype == torch.float32 and obs.is_contiguous() and zone_obs.is_contiguous()
        if out is None:
            out = torch.empty(B, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (B, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode(self.shape, B, obs.data_ptr(), zone_obs.data_ptr(),
                                                self.packed.data_ptr(), out.data_ptr(), self._status.data_ptr(),
                                                self._stream()))
        return out

    def pooled_from_state(self, env, out=None):
        """``pooled`` with the zone part of the input rows built from the env's STATE planes (crl_zone_encode_state)
        instead of read from ``env.zone_obs``: bit-identical to ``pooled(env.obs, env.zone_obs)`` after a step that
        wrote zone_obs, and the way to consume steps taken with ``env.write_zone_obs = False``."""
        B = env.num_envs
        assert env.spec.num_zones == self.num_zones and env.spec.zone_dim == self.zone_dim and self.obs_dim == 8
        if out is None:
            out = torch.empty(B, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (B, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_state(self.shape, env.cfg, env.state, env.obs.data_ptr(),
                                                      self.packed.data_ptr(), out.data_ptr(), self._status.data_ptr(),
                                                      self._stream()))
        return out

    def pooled_from_frames(self, obs, frames, out=None):
        """``pooled`` with the zone part of the rows built from a rollout's stored frames (``ZoneFrames``, any leading
        shape; obs of the same leading shape and 8 columns) by crl_zone_encode_frames: bit-identical to
        ``pooled(obs, frames.zone_obs())``."""
        assert frames.num_zones == self.num_zones and frames.zone_dim == self.zone_dim and self.obs_dim == 8
        rec = frames.flat_records()
        M = rec.shape[0]
        obs = obs.reshape(M, self.obs_dim)
        assert obs.dtype == torch.float32 and obs.is_contiguous()
        if out is None:
            out = torch.empty(M, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (M, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        xy, tm = frames.ptrs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_frames(self.shape, frames.cfg, M, obs.data_ptr(), rec.data_ptr(), xy, tm,
                                                       self.packed.data_ptr(), out.data_ptr(), self._status.data_ptr(),
                                                       self._stream()))
        return out

    def _workspace(self, B):
        """Scratch of crl_encoder_forward: the head kernel's bf16 operand images, one per 128 envs; None if the shape is
        not ZoneEnvModel's own (then the forward runs as two calls with an fp32 ``pooled`` in between)."""
        ws = self._ws.get(B)
        if ws is None:
            n = ctypes.c_int64()
            rc = self.lib.crl_encoder_workspace_bytes(self.shape, B, ctypes.byref(n))
            if rc == -4:                                   # CRL_ERR_UNSUPPORTED: not ZoneEnvModel's own shape
                ws = False
            else:
                _lib.check(rc)
                ws = torch.empty(n.value, dtype=torch.uint8, device=self.device)
            self._ws = {B: ws}                      # one batch size at a time
        return ws if ws is not False else None

    def _forward(self, obs, zone_obs=None, env=None, out=None, head=None):
        B = obs.shape[0]
        head = self.packed_head if head is None else head
        ws = self._workspace(B)
        if ws is None:
            pooled = self.pooled(obs, zone_obs) if env is None else self.pooled_from_state(env)
            return self._head(head, obs, pooled, out)
        if out is None:
            out = torch.empty(B, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (B, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        assert obs.shape == (B, self.obs_dim) and obs.dtype == torch.float32 and obs.is_contiguous()
        if env is None:
            assert zone_obs.shape == (B, self.num_zones, self.zone_dim) and zone_obs.dtype == torch.float32 and zone_obs.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_encoder_forward(
                self.shape, env.cfg if env is not None else None, env.state if env is not None else None, B, obs.data_ptr(),
                None if env is not None else zone_obs.data_ptr(), self.packed.data_ptr(), head.data_ptr(),
                ws.data_ptr(), out.data_ptr(), self._status.data_ptr(), self._stream()))
        return out

    def forward_from_state(self, env, out=None):
        """ZoneEnvModel.forward on the env's current observation without touching ``env.zone_obs``."""
        assert env.spec.num_zones == self.num_zones and env.spec.zone_dim == self.zone_dim and self.obs_dim == 8
        return self._forward(env.obs, env=env, out=out)

    def _head(self, packed, obs, pooled, out=None):
        B = obs.shape[0]
        if out is None:
            out = torch.empty(B, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (B, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_encoder_head(self.shape, B, obs.data_ptr(), pooled.data_ptr(), packed.data_ptr(),
                                                 out.data_ptr(), self._status.data_ptr(), self._stream()))
        return out

    def zone_embedding(self, obs, zone_obs, out=None):
        """mean_z zone_net_([obs, zone_obs[:, z]]) (env_model.py:73) = L3(pooled): the fused two-launch forward with the
        head weights [0 | W3]."""
        return self._forward(obs, zone_obs, out=out, head=self.packed_l3)

    # ---- precise mode: split-bf16 operands (three MMAs per product), fp32 biases; like for like with the fp32 module ----
    def _precise_image(self):
        if self._packed_precise is None:
            n = ctypes.c_int64()
            _lib.check(self.lib.crl_encoder_precise_packed_bytes(self.shape, ctypes.byref(n)))
            buf = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
            w1, b1, w2, b2 = self._keep[:4]
            with torch.cuda.device(self.device):
                _lib.check(self.lib.crl_encoder_pack_precise(self.shape, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                                             b2.data_ptr(), buf.data_ptr(), self._stream()))
            self._packed_precise = buf
        return self._packed_precise

    def pooled_precise(self, obs, zone_obs, out=None):
        """``pooled`` to fp32-level accuracy (crl_zone_encode_precise): ~1e-5 of the largest value against the fp32
        module instead of 3-5e-3, at ~7x the fast kernel's time (620 us at 65,536 PointTSP envs)."""
        B = obs.shape[0]
        assert obs.shape == (B, self.obs_dim) and zone_obs.shape == (B, self.num_zones, self.zone_dim)
        assert obs.dtype == zone_obs.dtype == torch.float32 and obs.is_contiguous() and zone_obs.is_contiguous()
        if out is None:
            out = torch.empty(B, self.hidden, dtype=torch.float32, device=self.device)
        assert out.shape == (B, self.hidden) and out.dtype == torch.float32 and out.is_contiguous()
        img = self._precise_image()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_precise(self.shape, B, obs.data_ptr(), zone_obs.data_ptr(), img.data_ptr(),
                                                        out.data_ptr(), self._status.data_ptr(), self._stream()))
        return out

    def _head_precise(self, key, w, b, obs, pooled):
        """An affine map of [obs, pooled] to fp32-level accuracy on the SAME tensor-core head kernel: it multiplies
        bf16(W) bf16(X), so three launches -- (W, X), (W - bf16 W, X), (W, X - bf16 X) -- add up to the split product
        W_hi X_hi + W_lo X_hi + W_hi X_lo; the bias rides in the first one (as its bf16 hi + lo pair).  No library GEMM."""
        imgs = self._precise_heads.get(key)
        if imgs is None:
            n = ctypes.c_int64()
            _lib.check(self.lib.crl_encoder_head_packed_bytes(self.shape, ctypes.byref(n)))
            r = lambda t: t.to(torch.bfloat16).to(torch.float32)
            zero = torch.zeros_like(b)
            imgs, keep = [], []
            for wi, bi in ((w, b), ((w - r(w)).contiguous(), zero), (w, zero)):
                buf = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
                with torch.cuda.device(self.device):
                    _lib.check(self.lib.crl_encoder_pack_head(self.shape, wi.data_ptr(), bi.data_ptr(), buf.data_ptr(), self._stream()))
                imgs.append(buf)
                keep.append((wi, bi))
            torch.cuda.current_stream(self.device).synchronize()       # the temporaries may go
            self._precise_heads[key] = imgs
        r = lambda t: t.to(torch.bfloat16).to(torch.float32)
        out = self._head(imgs[0], obs, pooled)
        out += self._head(imgs[1], obs, pooled)
        out += self._head(imgs[2], (obs - r(obs)).contiguous(), (pooled - r(pooled)).contiguous())
        return out

    def zone_embedding_precise(self, obs, zone_obs):
        """L3(pooled) to fp32-level accuracy: precise zone kernel + the split head (three launches of the head kernel)."""
        l3_w = torch.cat([torch.zeros(self.hidden, self.obs_dim, device=self.device), self.w3], dim=1).contiguous()
        return self._head_precise('l3', l3_w, self.b3, obs, self.pooled_precise(obs, zone_obs))

    def forward_precise(self, obs, zone_obs=None):
        """ZoneEnvModel.forward to fp32-level accuracy: precise zone kernel + the split head on the folded affine map."""
        if zone_obs is None:
            obs, zone_obs = obs['obs'], obs['zone_obs']
        return self._head_precise('fold', self.fold_w, self.fold_b, obs, self.pooled_precise(obs, zone_obs))

    def healthy(self):
        """False if a tensor-core completion wait ever expired (synchronises)."""
        return int(self._status.item()) == 0

    def __call__(self, obs, zone_obs=None):
        """ZoneEnvModel.forward: accepts the env's obs dict or the two tensors.  A dict that carries ``zone_frames``
        (Rollout(store='frames')) instead of ``zone_obs`` runs ``pooled_from_frames`` and the head kernel."""
        if zone_obs is None:
            if 'zone_frames' in obs:
                o = obs['obs'].reshape(-1, self.obs_dim)
                return self._head(self.packed_head, o, self.pooled_from_frames(o, obs['zone_frames']))
            obs, zone_obs = obs['obs'], obs['zone_obs']
        return self._forward(obs, zone_obs)


class _FusedCore:
    """The library calls behind FusedZoneEnvModel for one (obs_dim, zone_dim, hidden, num_zones): the packed weight
    image (one buffer, re-packed by every forward and backward from the weights they were given) and the backward's
    workspace (one batch size at a time)."""

    def __init__(self, obs_dim, zone_dim, hidden, num_zones, device):
        self.lib = _lib.load()
        self.device = device
        self.shape = _lib.CrlEncoderShape(obs_dim=obs_dim, zone_dim=zone_dim, hidden=hidden, num_zones=num_zones)
        n = ctypes.c_int64()
        _lib.check(self.lib.crl_encoder_packed_bytes(self.shape, ctypes.byref(n)))
        self.packed = torch.zeros(n.value, dtype=torch.uint8, device=device)
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self._ws = (None, None)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def pack(self, w1, b1, w2, b2):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_encoder_pack(self.shape, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                                 self.packed.data_ptr(), self._stream()))

    def pooled(self, obs, zone_obs):
        out = torch.empty(obs.shape[0], self.shape.hidden, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode(self.shape, obs.shape[0], obs.data_ptr(), zone_obs.data_ptr(),
                                                self.packed.data_ptr(), out.data_ptr(), self.status.data_ptr(),
                                                self._stream()))
        return out

    def _workspace(self, B):
        if self._ws[0] != B:
            n = ctypes.c_int64()
            with torch.cuda.device(self.device):
                _lib.check(self.lib.crl_encoder_backward_workspace_bytes(self.shape, B, ctypes.byref(n)))
            self._ws = (B, torch.empty(n.value, dtype=torch.uint8, device=self.device))
        return self._ws[1]

    def _grads(self):
        h, in_dim = self.shape.hidden, self.shape.obs_dim + self.shape.zone_dim
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=self.device)
        return f(h, in_dim), f(h), f(h, h), f(h)

    def backward(self, obs, zone_obs, grad_pooled):
        B = obs.shape[0]
        ws = self._workspace(B)
        dw1, db1, dw2, db2 = self._grads()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_backward(
                self.shape, B, obs.data_ptr(), zone_obs.data_ptr(), self.packed.data_ptr(), grad_pooled.data_ptr(),
                ws.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), db2.data_ptr(),
                self.status.data_ptr(), self._stream()))
        return dw1, db1, dw2, db2

    # the same from stored frames (records (M, 4) int32 and the rollout's layout table)
    def pooled_frames(self, obs, records, frames):
        out = torch.empty(obs.shape[0], self.shape.hidden, dtype=torch.float32, device=self.device)
        xy, tm = frames.ptrs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_frames(self.shape, frames.cfg, obs.shape[0], obs.data_ptr(),
                                                       records.data_ptr(), xy, tm, self.packed.data_ptr(), out.data_ptr(),
                                                       self.status.data_ptr(), self._stream()))
        return out

    def backward_frames(self, obs, records, frames, grad_pooled):
        B = obs.shape[0]
        ws = self._workspace(B)
        dw1, db1, dw2, db2 = self._grads()
        xy, tm = frames.ptrs()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.crl_zone_encode_backward_frames(
                self.shape, frames.cfg, B, obs.data_ptr(), records.data_ptr(), xy, tm, self.packed.data_ptr(),
                grad_pooled.data_ptr(), ws.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), db2.data_ptr(),
                self.status.data_ptr(), self._stream()))
        return dw1, db1, dw2, db2


class _FusedPooled(torch.autograd.Function):
    """pooled = mean_z relu(W2 relu(W1 [obs, zone_obs[:, z]] + b1) + b2) with gradients for W1, b1, W2, b2."""

    @staticmethod
    def forward(ctx, core, obs, zone_obs, w1, b1, w2, b2):
        if obs.requires_grad or zone_obs.requires_grad:
            raise RuntimeError('FusedZoneEnvModel: gradients with respect to obs / zone_obs are not computed; '
                               'detach the inputs')
        core.pack(w1, b1, w2, b2)
        ctx.core = core
        ctx.save_for_backward(obs, zone_obs, w1, b1, w2, b2)    # the version counters catch an in-place update
        return core.pooled(obs, zone_obs)

    @staticmethod
    def backward(ctx, grad_pooled):
        obs, zone_obs, w1, b1, w2, b2 = ctx.saved_tensors
        ctx.core.pack(w1, b1, w2, b2)                             # the image of exactly the weights the forward used
        dw1, db1, dw2, db2 = ctx.core.backward(obs, zone_obs, grad_pooled.contiguous())
        return None, None, None, dw1, db1, dw2, db2


class _FusedPooledFrames(torch.autograd.Function):
    """_FusedPooled with the zone rows built from stored frames (crl_zone_encode_frames / _backward_frames)."""

    @staticmethod
    def forward(ctx, core, frames, obs, records, w1, b1, w2, b2):
        if obs.requires_grad:
            raise RuntimeError('FusedZoneEnvModel: gradients with respect to obs are not computed; detach the inputs')
        core.pack(w1, b1, w2, b2)
        ctx.core, ctx.frames = core, frames
        ctx.save_for_backward(obs, records, w1, b1, w2, b2)
        return core.pooled_frames(obs, records, frames)

    @staticmethod
    def backward(ctx, grad_pooled):
        obs, records, w1, b1, w2, b2 = ctx.saved_tensors
        ctx.core.pack(w1, b1, w2, b2)
        dw1, db1, dw2, db2 = ctx.core.backward_frames(obs, records, ctx.frames, grad_pooled.contiguous())
        return None, None, None, None, dw1, db1, dw2, db2


class FusedZoneEnvModel(nn.Module):
    """The reference's ZoneEnvModel (env_model.py:48-79) with its (B N)-row part forward and backward on the tensor
    cores.  ``forward(obs)`` takes the env's obs dict or an object with ``.obs`` / ``.zone_obs`` (the reference's DictList)
    and returns ``combine_net_([obs, zone_net_[4](pooled)])``."""

    def __init__(self, obs_dim, zone_dim, num_zones, hidden=185, device='cuda:0'):
        super().__init__()
        if not torch.cuda.is_available():
            raise RuntimeError('FusedZoneEnvModel needs a CUDA device (sm_100a); there is no CPU fallback')
        self.obs_dim, self.zone_dim, self.num_zones, self.hidden = int(obs_dim), int(zone_dim), int(num_zones), int(hidden)
        self.zone_net_ = nn.Sequential(nn.Linear(obs_dim + zone_dim, hidden), nn.ReLU(), nn.Linear(hidden, hidden),
                                       nn.ReLU(), nn.Linear(hidden, hidden))
        self.combine_net_ = nn.Linear(obs_dim + hidden, hidden)
        self.to(device)
        self._core = _FusedCore(self.obs_dim, self.zone_dim, self.hidden, self.num_zones, torch.device(device))

    def pooled(self, obs, zone_obs):
        B = obs.shape[0]
        assert obs.shape == (B, self.obs_dim) and zone_obs.shape == (B, self.num_zones, self.zone_dim)
        assert obs.dtype == zone_obs.dtype == torch.float32
        l1, l2 = self.zone_net_[0], self.zone_net_[2]
        return _FusedPooled.apply(self._core, obs.contiguous(), zone_obs.contiguous(),
                                  l1.weight.contiguous(), l1.bias.contiguous(), l2.weight.contiguous(), l2.bias.contiguous())

    def pooled_from_frames(self, obs, frames):
        """``pooled`` of rows built from stored frames (``ZoneFrames``; Rollout(store='frames')), forward and backward:
        the same numbers as ``pooled(obs, frames.zone_obs())`` without the rows ever being materialised.  The frames stay
        valid until the rollout's next ``begin()``: run the backward before that."""
        assert frames.num_zones == self.num_zones and frames.zone_dim == self.zone_dim and self.obs_dim == 8
        records = frames.flat_records()
        obs = obs.reshape(records.shape[0], self.obs_dim)
        assert obs.dtype == torch.float32
        l1, l2 = self.zone_net_[0], self.zone_net_[2]
        return _FusedPooledFrames.apply(self._core, frames, obs.contiguous(), records, l1.weight.contiguous(),
                                        l1.bias.contiguous(), l2.weight.contiguous(), l2.bias.contiguous())

    def forward(self, obs):
        """``obs``: a dict / DictList with ``obs`` and either ``zone_obs`` or ``zone_frames`` (Rollout(store='frames'))."""
        get = (lambda k: obs.get(k)) if isinstance(obs, dict) else (lambda k: getattr(obs, k, None))
        o, z, fr = get('obs'), get('zone_obs'), get('zone_frames')
        if z is None and fr is not None:
            o = o.reshape(-1, self.obs_dim)
            pooled = self.pooled_from_frames(o, fr)
        else:
            pooled = self.pooled(o, z)
        return self.combine_net_(torch.cat([o, self.zone_net_[4](pooled)], dim=-1))

    def healthy(self):
        """False if a tensor-core completion wait ever expired (synchronises)."""
        return int(self._core.status.item()) == 0
