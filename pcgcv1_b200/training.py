"""One training step of the hyperprior model on the GPU (SURVEY.md 8a row a22 / BASELINE config 5).

Mirrors ``train_hyper.py:184-214``: forward with "noise" quantisation in both entropy models, rate-distortion loss
``alpha * (beta * empty + full) + delta * bpp_y + gamma * bpp_z`` with the BCE occupancy loss of ``loss.py:8-33``, gradients of
every trainable variable (analysis / synthesis / hyper encoder / hyper decoder kernels and biases, EntropyBottleneck matrices /
biases / factors) and an Adam update (``tf.train.AdamOptimizer`` arithmetic).

Every computation is a C-ABI call into libpcgc_b200.so (csrc/train.cu, conv_ffma.cu, entropy.cu): exact FP32, fixed reduction
orders.  torch is the buffer allocator and -- through ``torch.autograd.Function`` -- the TAPE that orders the backward calls;
no torch operator does model arithmetic.  The reference draws its noise from an unseeded TF stream; here the noise is a
seeded Philox stream (``seed`` per step), which the oracle (oracle/train.py) reproduces bit for bit.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional

import numpy as np
import torch

from . import netspec, runtime, weights as W

_NETS = ("analysis_transform", "synthesis_transform", "hyper_encoder", "hyper_decoder")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class _Ops:
    """Thin wrappers: torch tensors in, C ABI underneath."""

    def __init__(self, codec: runtime.Codec):
        self.c = codec
        self.lib = codec.lib

    def _go(self, rc):
        self.c._check(rc)

    def conv_forward(self, x, w, b, l: netspec.Layer):
        B, n = x.shape[0], x.shape[1]
        m = n * l.stride if l.transposed else n // l.stride
        out = torch.empty((B, m, m, m, l.cout), dtype=torch.float32, device=x.device)
        self.c._stream()
        self._go(self.lib.pcgc_train_conv_forward(self.c.ctx, x.data_ptr(), B, n, l.cin, l.cout, l.k, l.stride, int(l.transposed), w.data_ptr(), _ptr(b),
                                                  int(l.relu), out.data_ptr()))
        return out

    def conv_dgrad(self, g, w, l: netspec.Layer, n: int):
        B = g.shape[0]
        dx = torch.empty((B, n, n, n, l.cin), dtype=torch.float32, device=g.device)
        self.c._stream()
        self._go(self.lib.pcgc_train_conv_dgrad(self.c.ctx, g.data_ptr(), B, n, l.cin, l.cout, l.k, l.stride, int(l.transposed), w.data_ptr(), dx.data_ptr()))
        return dx

    def conv_wgrad(self, x, g, w, l: netspec.Layer):
        B, n = x.shape[0], x.shape[1]
        dw = torch.empty_like(w)
        db = torch.empty(l.cout, dtype=torch.float32, device=x.device) if l.bias else None
        self.c._stream()
        self._go(self.lib.pcgc_train_conv_wgrad(self.c.ctx, x.data_ptr(), g.data_ptr(), B, n, l.cin, l.cout, l.k, l.stride, int(l.transposed),
                                                dw.data_ptr(), _ptr(db)))
        return dw, db

    def relu_backward(self, g, y):
        out = torch.empty_like(g)
        self.c._stream()
        self._go(self.lib.pcgc_train_relu_backward(self.c.ctx, g.data_ptr(), y.data_ptr(), g.numel(), out.data_ptr()))
        return out


class _Conv(torch.autograd.Function):
    """One Keras Conv3D / Conv3DTranspose layer: conv -> bias -> activation."""

    @staticmethod
    def forward(ctx, x, w, b, ops: _Ops, layer: netspec.Layer):
        x = x.contiguous()
        out = ops.conv_forward(x, w, b, layer)
        ctx.save_for_backward(x, w, out)
        ctx.ops, ctx.layer, ctx.has_bias = ops, layer, b is not None
        return out

    @staticmethod
    def backward(ctx, g):
        x, w, out = ctx.saved_tensors
        ops, l = ctx.ops, ctx.layer
        g = g.contiguous()
        if l.relu:
            g = ops.relu_backward(g, out)
        dx = ops.conv_dgrad(g, w, l, x.shape[1]) if ctx.needs_input_grad[0] else None
        dw, db = ops.conv_wgrad(x, g, w, l)
        return dx, dw, (db if ctx.has_bias else None), None, None


class _VrnMerge(torch.autograd.Function):
    """out = relu(x + concat[t12, t23]) (model_voxception.py:64-67)."""

    @staticmethod
    def forward(ctx, x, t12, t23, ops: _Ops):
        x, t12, t23 = x.contiguous(), t12.contiguous(), t23.contiguous()
        out = torch.empty_like(x)
        c = x.shape[-1]
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_vrn_merge(ops.c.ctx, x.data_ptr(), t12.data_ptr(), t23.data_ptr(), x.numel() // c, c, out.data_ptr()))
        ctx.save_for_backward(out)
        ctx.ops, ctx.h = ops, t12.shape
        return out

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        ops = ctx.ops
        g = g.contiguous()
        c = out.shape[-1]
        gx = torch.empty_like(out)
        g12 = torch.empty(ctx.h, dtype=torch.float32, device=out.device)
        g23 = torch.empty(ctx.h, dtype=torch.float32, device=out.device)
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_vrn_merge_backward(ops.c.ctx, g.data_ptr(), out.data_ptr(), out.numel() // c, c, gx.data_ptr(), g12.data_ptr(), g23.data_ptr()))
        return gx, g12, g23, None


class _AbsFloor(torch.autograd.Function):
    """scale = max(|s|, lower_bound) (model_voxception.py:308 + train_hyper.py:191)."""

    @staticmethod
    def forward(ctx, s, floor_v: float, ops: _Ops):
        s = s.contiguous()
        out = torch.empty_like(s)
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_abs_floor(ops.c.ctx, s.data_ptr(), s.numel(), floor_v, out.data_ptr()))
        ctx.save_for_backward(s)
        ctx.ops, ctx.floor_v = ops, floor_v
        return out

    @staticmethod
    def backward(ctx, g):
        (s,) = ctx.saved_tensors
        ops = ctx.ops
        g = g.contiguous()
        out = torch.empty_like(s)
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_abs_floor_backward(ops.c.ctx, g.data_ptr(), s.data_ptr(), s.numel(), ctx.floor_v, out.data_ptr()))
        return out, None, None


class _LaplaceRate(torch.autograd.Function):
    """SymmetricConditional(y, loc, scale, training=True): returns y_t = y + noise; its backward adds the gradient of the rate
    term ``coef * sum(log max(p, bound))`` (coef = delta / (-ln 2 * num_points), known on the host) to what flows back from the
    synthesis transform.  ``stats['logsum_y']`` receives sum(log p) as a device scalar for the loss report."""

    @staticmethod
    def forward(ctx, y, loc, scale, coef: float, seed: int, bound: float, ops: _Ops, stats: dict):
        c = ops.c
        B = y.shape[0]
        y2, l2, s2 = y.contiguous().reshape(B, -1), loc.contiguous().reshape(B, -1), scale.contiguous().reshape(B, -1)
        c.set_quantize_mode(True, seed)
        try:
            y_t, _, bits, _ = c.laplace(y2, l2, s2, bound, want_p=False, want_bits=True)
        finally:
            c.set_quantize_mode(False)
        stats["bits_y"] = bits                                           # per cube: -sum(log2 p)
        ctx.save_for_backward(y_t, l2, s2)
        ctx.ops, ctx.coef, ctx.bound, ctx.shape = ops, coef, bound, y.shape
        return y_t.reshape(y.shape)

    @staticmethod
    def backward(ctx, g):
        y_t, loc, scale = ctx.saved_tensors
        ops = ctx.ops
        gy, gl, gs = torch.empty_like(y_t), torch.empty_like(y_t), torch.empty_like(y_t)
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_laplace_backward(ops.c.ctx, y_t.data_ptr(), loc.data_ptr(), scale.data_ptr(), y_t.numel(), ctx.bound, ctx.coef,
                                                    gy.data_ptr(), gl.data_ptr(), gs.data_ptr()))
        gy = _axpy(ops, gy, g.contiguous().reshape(gy.shape))
        return gy.reshape(ctx.shape), gl.reshape(ctx.shape), gs.reshape(ctx.shape), None, None, None, None, None


class _FactorizedRate(torch.autograd.Function):
    """EntropyBottleneck(z, training=True) from its raw variables: returns z_t; backward adds the rate term's gradient w.r.t. z
    and produces the gradients of the matrices / biases / factors."""

    @staticmethod
    def forward(ctx, z, matrices, biases, factors, coef: float, seed: int, bound: float, ops: _Ops, stats: dict):
        c = ops.c
        z = z.contiguous()
        Cz = z.shape[-1]
        z_t = torch.empty_like(z)
        logsum = torch.empty(1, dtype=torch.float64, device=z.device)
        c._stream()
        ops._go(ops.lib.pcgc_train_factorized_forward(c.ctx, matrices.data_ptr(), biases.data_ptr(), factors.data_ptr(), Cz, z.data_ptr(),
                                                      z.numel() // Cz, int(seed) & 0xFFFFFFFFFFFFFFFF, bound, z_t.data_ptr(), logsum.data_ptr()))
        stats["logsum_z"] = logsum
        ctx.save_for_backward(z_t, matrices, biases, factors)
        ctx.ops, ctx.coef, ctx.bound = ops, coef, bound
        return z_t

    @staticmethod
    def backward(ctx, g):
        z_t, m, b, f = ctx.saved_tensors
        ops = ctx.ops
        Cz = z_t.shape[-1]
        gz, gm, gb, gf = torch.empty_like(z_t), torch.empty_like(m), torch.empty_like(b), torch.empty_like(f)
        ops.c._stream()
        ops._go(ops.lib.pcgc_train_factorized_backward(ops.c.ctx, m.data_ptr(), b.data_ptr(), f.data_ptr(), Cz, z_t.data_ptr(), z_t.numel() // Cz,
                                                       ctx.bound, ctx.coef, gz.data_ptr(), gm.data_ptr(), gb.data_ptr(), gf.data_ptr()))
        gz = _axpy(ops, gz, g.contiguous())
        return gz, gm, gb, gf, None, None, None, None, None


def _axpy(ops: _Ops, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a + b on the device (gradient accumulation where two paths meet inside one Function).  A tensor add is buffer plumbing of
    the tape, the same operation torch.autograd itself performs when a tensor feeds two consumers."""
    return a.add_(b)


class _Trainer:
    """What every training step shares: the trainable variables (Keras names / layouts) as device buffers, the layer graph of
    the transforms, the occupancy loss, Adam, the data-parallel all-reduce and the export to the weight-file form.

    ``nets`` are the top-level checkpoint keys of the transforms this model trains; ``bottlenecks`` maps the checkpoint prefix of
    every EntropyBottleneck it trains (``estimator/``, ``estimator_y/``) to its channel count.  A bottleneck's matrices /
    biases / factors are held concatenated in the ``pcgc_load_bottleneck`` order under ``<prefix>matrix|bais|factor``."""

    def __init__(self, codec, weights, model, nets, bottlenecks, alpha, beta, delta, lr, likelihood_bound, distortion, focal_gamma,
                 focal_alpha):
        if distortion not in ("bce", "focal"):
            raise ValueError("distortion must be 'bce' or 'focal', got %r" % (distortion,))
        self.distortion, self.focal_gamma, self.focal_alpha = distortion, float(focal_gamma), float(focal_alpha)
        self.model, self.nets, self.bottlenecks = model, tuple(nets), dict(bottlenecks)
        self.codec = codec or runtime.get_codec(model, "")
        self.ops = _Ops(self.codec)
        w = weights if weights is not None else W.synthetic_weights(model)
        dev = self.codec.dev
        self.params: Dict[str, torch.Tensor] = {}
        for net in self.nets:
            for l in netspec.NETS[(model, net)]:
                for kind in ("kernel", "bias"):
                    key = "%s/%s/%s" % (net, l.name, kind)
                    if key in w:
                        self.params[key] = torch.tensor(np.ascontiguousarray(w[key], dtype=np.float32), device=dev, requires_grad=True)
        for prefix in self.bottlenecks:
            cat = lambda name: np.concatenate([np.asarray(w["%s%s_%d" % (prefix, name, i)], np.float32).reshape(-1) for i in range(4)])
            for name in ("matrix", "bais", "factor"):
                self.params[prefix + name] = torch.tensor(cat(name), device=dev, requires_grad=True)
        self.alpha, self.beta, self.delta = float(alpha), float(beta), float(delta)
        self.lr, self.likelihood_bound = float(lr), float(likelihood_bound)
        self.step_count = 0
        self.adam_m = {k: torch.zeros_like(v) for k, v in self.params.items()}
        self.adam_v = {k: torch.zeros_like(v) for k, v in self.params.items()}

    # ---- the graph (models/model_voxception.py, models/model_simple.py) ---------------------------------------------------
    def _conv(self, x, net: str, l: netspec.Layer):
        return _Conv.apply(x, self.params["%s/%s/kernel" % (net, l.name)], self.params.get("%s/%s/bias" % (net, l.name)), self.ops, l)

    def _run(self, net: str, x):
        table = netspec.NETS[(self.model, net)]
        layers = {l.name: l for l in table}
        names = [l.name for l in table]
        i = 0
        while i < len(names):
            n = names[i]
            if n.endswith("_conv1_1"):                                   # a _VoxceptionResNet block: 5 layers in table order
                p = n[:-len("_conv1_1")]
                t11 = self._conv(x, net, layers[p + "_conv1_1"])
                t12 = self._conv(t11, net, layers[p + "_conv1_2"])
                t21 = self._conv(x, net, layers[p + "_conv2_1"])
                t22 = self._conv(t21, net, layers[p + "_conv2_2"])
                t23 = self._conv(t22, net, layers[p + "_conv2_3"])
                x = _VrnMerge.apply(x, t12, t23, self.ops)
                i += 5
            else:
                x = self._conv(x, net, layers[n])
                i += 1
        return x

    def _begin(self, cubes):
        """-> (label uint8, x float32, num_points) on the device; clears every gradient."""
        c = self.codec
        label = c.to_device(cubes, torch.uint8)
        x = torch.empty(label.shape, dtype=torch.float32, device=c.dev)
        x.copy_(label)                                                    # dtype conversion of the input buffer
        num_points = int(np.count_nonzero(runtime.unwrap(cubes))) if not isinstance(cubes, torch.Tensor) else int(label.count_nonzero())
        for p in self.params.values():
            p.grad = None
        return label, x, num_points

    def _distortion_backward(self, x_t, label):
        """Occupancy loss sums on the device; its gradient seeds the backward pass.  -> {"bce_sums" | "focal_sums": sums}."""
        c = self.codec
        g = torch.empty_like(x_t)
        c._stream()
        if self.distortion == "focal":
            sums = torch.empty(2, dtype=torch.float64, device=c.dev)
            c._check(c.lib.pcgc_train_focal(c.ctx, x_t.data_ptr(), label.data_ptr(), x_t.numel(), self.focal_gamma, self.focal_alpha, sums.data_ptr()))
            c._check(c.lib.pcgc_train_focal_backward(c.ctx, x_t.data_ptr(), label.data_ptr(), x_t.numel(), self.focal_gamma, self.focal_alpha, self.alpha,
                                                     g.data_ptr()))
        else:
            sums = torch.empty(4, dtype=torch.float64, device=c.dev)
            c._check(c.lib.pcgc_train_bce(c.ctx, x_t.data_ptr(), label.data_ptr(), x_t.numel(), sums.data_ptr()))
            c._check(c.lib.pcgc_train_bce_backward(c.ctx, x_t.data_ptr(), label.data_ptr(), x_t.numel(), sums.data_ptr(), self.alpha * self.beta,
                                                   self.alpha, g.data_ptr()))
        x_t.backward(g)
        return {"bce_sums" if self.distortion == "bce" else "focal_sums": sums}

    def _distortion_terms(self, out) -> Dict[str, float]:
        """Host values of the occupancy loss: its parts and ``distortion`` (one synchronisation)."""
        if "focal_sums" in out:
            s = out["focal_sums"].cpu().numpy()
            return {"focal_full": float(s[0]), "focal_empty": float(s[1]), "distortion": float(s[0] + s[1])}
        s = out["bce_sums"].cpu().numpy()
        zeros, ones = s[0] / max(s[2], 1.0), s[1] / max(s[3], 1.0)
        return {"zeros": float(zeros), "ones": float(ones), "distortion": float(self.beta * zeros + ones)}

    def adam_step(self, beta1=0.9, beta2=0.999, eps=1e-8):
        """tf.train.AdamOptimizer.apply_gradients: lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t); p -= lr_t * m / (sqrt(v) + eps)."""
        c = self.codec
        self.step_count += 1
        t = self.step_count
        lr_t = self.lr * math.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)
        c._stream()
        for k, p in self.params.items():
            if p.grad is None:
                continue
            g = p.grad.contiguous()
            c._check(c.lib.pcgc_train_adam(c.ctx, p.data_ptr(), g.data_ptr(), self.adam_m[k].data_ptr(), self.adam_v[k].data_ptr(), p.numel(), lr_t, beta1, beta2,
                                           eps))

    def allreduce_gradients(self, group=None):
        """Data-parallel training (SURVEY.md 8f rank 4): average the gradients over the ranks of a torch.distributed group
        (NCCL over NVLink) -- ONE all-reduce of a flat buffer, then scattered back into the per-variable gradients."""
        import torch.distributed as dist
        if not dist.is_initialized() or dist.get_world_size(group) == 1:
            return
        keys = [k for k, p in self.params.items() if p.grad is not None]
        flat = torch.cat([self.params[k].grad.reshape(-1) for k in keys])
        dist.all_reduce(flat, group=group)
        flat.div_(dist.get_world_size(group))
        o = 0
        for k in keys:
            g = self.params[k].grad
            g.copy_(flat[o:o + g.numel()].view_as(g))
            o += g.numel()

    def train_step(self, cubes, seed: int = 0, group=None):
        out = self.forward_backward(cubes, seed)
        self.allreduce_gradients(group)
        self.adam_step()
        return out

    def export_weights(self) -> Dict[str, np.ndarray]:
        """Back to the weight-file form (Keras names; bottleneck variables split into <prefix>matrix_i / bais_i / factor_i)."""
        out = {k: v.detach().cpu().numpy() for k, v in self.params.items() if not k.startswith(tuple(self.bottlenecks))}
        for prefix, Cz in self.bottlenecks.items():
            shapes = {"matrix": [(Cz, 3, 1), (Cz, 3, 3), (Cz, 3, 3), (Cz, 1, 3)], "bais": [(Cz, 3, 1)] * 3 + [(Cz, 1, 1)],
                      "factor": [(Cz, 3, 1)] * 3 + [(Cz, 1, 1)]}
            for name, shp in shapes.items():
                flat = self.params[prefix + name].detach().cpu().numpy()
                o = 0
                for i, s in enumerate(shp):
                    n = int(np.prod(s))
                    out["%s%s_%d" % (prefix, name, i)] = flat[o:o + n].reshape(s).copy()
                    o += n
        return out


class HyperTrainer(_Trainer):
    """The hyperprior model (Voxception transforms, hyper encoder / decoder, EntropyBottleneck on z, conditional model on y)."""

    def __init__(self, codec: Optional[runtime.Codec] = None, weights: Optional[Dict[str, np.ndarray]] = None, alpha=0.75, beta=3.0, gamma=1.0,
                 delta=1.0, lr=1e-5, lower_bound=1e-9, likelihood_bound=1e-9, distortion="bce", focal_gamma=2.0, focal_alpha=0.9):
        """``distortion``: "bce" = ``get_bce_loss`` as ``train_hyper.py:199-203`` calls it (beta * empty + full); "focal" =
        ``get_focal_loss`` (``loss.py:83-93``, gamma 2, alpha 0.9, a SUM over the batch) on sigmoid(x_tilde) -- the reference
        defines it but neither train script calls it; BASELINE config 5 names it, so it is selectable and D = the focal sum."""
        super().__init__(codec, weights, "voxception", _NETS, {"estimator/": netspec.HYPER_CHANNELS}, alpha, beta, delta, lr, likelihood_bound,
                         distortion, focal_gamma, focal_alpha)
        self.gamma, self.lower_bound = float(gamma), float(lower_bound)

    def _hyper_decoder(self, z_t):
        layers = {l.name: l for l in netspec.NETS[("voxception", "hyper_decoder")]}
        f = self._conv(z_t, "hyper_decoder", layers["deconv1"])
        f = self._conv(f, "hyper_decoder", layers["deconv2"])
        f = self._conv(f, "hyper_decoder", layers["deconv3"])
        return self._conv(f, "hyper_decoder", layers["deconv4_1"]), self._conv(f, "hyper_decoder", layers["deconv4_2"])

    def forward_backward(self, cubes, seed: int = 0):
        """cubes uint8 [B,64,64,64,1] (host or device) -> dict of loss terms (device scalars) with .grad set on every parameter."""
        ops = self.ops
        label, x, num_points = self._begin(cubes)
        stats: dict = {}
        coef_y = self.delta / (-math.log(2.0) * num_points)
        coef_z = self.gamma / (-math.log(2.0) * num_points)
        y = self._run("analysis_transform", x)
        z = self._run("hyper_encoder", y)
        z_t = _FactorizedRate.apply(z, self.params["estimator/matrix"], self.params["estimator/bais"], self.params["estimator/factor"], coef_z, seed,
                                    self.likelihood_bound, ops, stats)
        loc, s_raw = self._hyper_decoder(z_t)
        scale = _AbsFloor.apply(s_raw, self.lower_bound, ops)
        y_t = _LaplaceRate.apply(y, loc, scale, coef_y, seed, self.likelihood_bound, ops, stats)
        x_t = self._run("synthesis_transform", y_t)
        out = self._distortion_backward(x_t, label)
        out.update({"bits_y": stats["bits_y"], "logsum_z": stats["logsum_z"], "num_points": num_points, "x_tilde": x_t.detach()})
        return out

    def loss_terms(self, out) -> Dict[str, float]:
        """Host values of the step's loss terms (one synchronisation)."""
        n = out["num_points"]
        bpp_y = float(out["bits_y"].sum().item()) / n
        bpp_z = float(out["logsum_z"].item()) / (-math.log(2.0) * n)
        t = self._distortion_terms(out)
        t.update({"bpp_ae": bpp_y, "bpp_hyper": bpp_z, "loss": float(self.alpha * t["distortion"] + self.delta * bpp_y + self.gamma * bpp_z)})
        return t


class FactorizedTrainer(_Trainer):
    """The factorized-prior model: analysis -> ``EntropyBottleneck(y, training=True)`` -> synthesis, for ``model_simple`` (32-channel
    y, the ``estimator/*`` variables) or the Voxception transforms (16-channel y, ``estimator_y/*``: the slot the codec's factorized
    path loads; no hyper nets).

    The loss is ``alpha * (beta * empty + full) + delta * bpp_y`` with the BCE (or ``alpha * focal`` with ``distortion="focal"``):
    the hyperprior step of ``HyperTrainer`` with its hyperprior terms removed.  The reference's ``train_factorized.py`` is not
    available, so this is this project's definition of the factorized training loss, not a parity claim.  The noise on y is the
    factorized training stream of ``pcgc_train_factorized_forward`` seeded with the step's ``seed`` (the stream z draws from in
    the hyperprior step)."""

    def __init__(self, codec: Optional[runtime.Codec] = None, weights: Optional[Dict[str, np.ndarray]] = None, model: str = "simple", alpha=0.75,
                 beta=3.0, delta=1.0, lr=1e-5, likelihood_bound=1e-9, distortion="bce", focal_gamma=2.0, focal_alpha=0.9):
        if model not in ("simple", "voxception"):
            raise ValueError("model must be 'simple' or 'voxception', got %r" % (model,))
        prefix = "estimator/" if model == "simple" else "estimator_y/"
        super().__init__(codec or runtime.get_codec(model, ""), weights, model, ("analysis_transform", "synthesis_transform"),
                         {prefix: netspec.LATENT_CHANNELS[model]}, alpha, beta, delta, lr, likelihood_bound, distortion, focal_gamma, focal_alpha)
        if self.codec.model != model:
            raise ValueError("the codec runs model %r, the trainer %r" % (self.codec.model, model))
        self.prefix = prefix

    def forward_backward(self, cubes, seed: int = 0):
        """cubes uint8 [B,64,64,64,1] (host or device) -> dict of loss terms (device scalars) with .grad set on every parameter."""
        label, x, num_points = self._begin(cubes)
        stats: dict = {}
        coef_y = self.delta / (-math.log(2.0) * num_points)
        y = self._run("analysis_transform", x)
        p = self.prefix
        y_t = _FactorizedRate.apply(y, self.params[p + "matrix"], self.params[p + "bais"], self.params[p + "factor"], coef_y, seed,
                                    self.likelihood_bound, self.ops, stats)
        x_t = self._run("synthesis_transform", y_t)
        out = self._distortion_backward(x_t, label)
        out.update({"logsum_y": stats["logsum_z"], "num_points": num_points, "x_tilde": x_t.detach()})
        return out

    def loss_terms(self, out) -> Dict[str, float]:
        """Host values of the step's loss terms (one synchronisation)."""
        bpp_y = float(out["logsum_y"].item()) / (-math.log(2.0) * out["num_points"])
        t = self._distortion_terms(out)
        t.update({"bpp_ae": bpp_y, "loss": float(self.alpha * t["distortion"] + self.delta * bpp_y)})
        return t
