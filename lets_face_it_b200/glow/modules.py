"""Flow primitives with the reference's module API, backed by the sm_100a kernels.

Same class names, constructor signatures, parameter/buffer names and shapes as
`code/glow_pytorch/glow/modules.py` of the reference (so its checkpoints load, SURVEY.md §5), but
`forward` calls liblfi_b200.so through `_cabi` — CUDA tensors only, no torch fallback.
Gradients flow through the fused `SeqGlow.forward` path, through `FlowStep / FlowNet / Glow.forward` (one autograd node
per flow step and frame, models.py: `_FlowStepFn`) and through the stand-alone `ActNorm2d / InvertibleConv1x1 / LinearZeros`
calls below, as in the reference, whose modules are plain autograd modules.  A call takes the autograd path when grad mode
is on and its input or one of its parameters requires grad; otherwise the inference path runs.  Both paths launch the same
forward kernels, so a forward value does not depend on grad mode.  The parameter-only log-det terms (C * sum(logs),
C * sum(log_s), C * slogdet(W)) are computed by torch, which then owns their gradients.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg
import torch
import torch.nn as nn

from .. import _cabi as cabi


def _f32c(t, device=None):
    t = t.detach()
    if device is not None:
        t = t.to(device)
    return t.to(torch.float32).contiguous()


def _f32g(t, device):
    """`_f32c` without the detach: the move / cast stays on the autograd graph (no copy when `t` already fits)."""
    return t.to(device=device, dtype=torch.float32).contiguous()


def _needs_grad(*ts):
    """The dispatch rule of every module here (and of FlowStep.forward): autograd when grad mode is on and a tensor involved
    requires grad."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _gemm(transA, transB, M, N, K, a, b, c):
    """c = op(a) op(b) in fp32 (lfi_gemm, no epilogue: every output element is one thread's fixed-order sum)."""
    lda = M if transA else K
    ldb = K if transB else N
    cabi.check(cabi.lib().lfi_gemm(cabi.GEMM_FP32, transA, transB, M, N, K, cabi.ptr(a), lda, 0, cabi.ptr(b), ldb, 0, cabi.ptr(c), N, 0,
                                   None, 0, None, 0, 0, 1, 0, None, 0, cabi.stream_ptr()), "lfi_gemm")
    return c


def _actnorm(x, bias, logs, reverse):
    y = torch.empty_like(x)
    B, C = x.shape
    cabi.check(cabi.lib().lfi_actnorm(cabi.ptr(x), cabi.ptr(bias), cabi.ptr(logs), cabi.ptr(y), B, C, int(bool(reverse)), cabi.stream_ptr()),
               "lfi_actnorm")
    return y


class _ActNormFn(torch.autograd.Function):
    """ActNorm2d on [B, C] under autograd: forward = lfi_actnorm, backward = lfi_actnorm_bwd."""

    @staticmethod
    def forward(ctx, x, bias, logs, reverse):
        y = _actnorm(x, bias.detach(), logs.detach(), reverse)
        ctx.reverse = reverse
        ctx.save_for_backward(x, y, bias, logs)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, _, logs = ctx.saved_tensors
        B, C = x.shape
        dy = dy.to(torch.float32).contiguous()
        dx = torch.empty_like(x)
        dbias = torch.empty(1, C, dtype=torch.float32, device=x.device)
        dlogs = torch.empty(1, C, dtype=torch.float32, device=x.device)
        cabi.check(cabi.lib().lfi_actnorm_bwd(cabi.ptr(x), cabi.ptr(y), cabi.ptr(logs), cabi.ptr(dy), cabi.ptr(dx), cabi.ptr(dbias),
                                              cabi.ptr(dlogs), B, C, int(ctx.reverse), cabi.stream_ptr()), "lfi_actnorm_bwd")
        return dx, dbias, dlogs, None


def _matmul(x, w):
    B, C = x.shape
    z = torch.empty(B, w.shape[1], dtype=torch.float32, device=x.device)
    cabi.check(cabi.lib().lfi_matmul(cabi.ptr(x), cabi.ptr(w), None, cabi.ptr(z), B, w.shape[1], C, 0, cabi.stream_ptr()), "lfi_matmul")
    return z


class _MatmulFn(torch.autograd.Function):
    """z = x @ W (InvertibleConv1x1.forward, modules.py:186) under autograd: dx = dz W^T, dW = x^T dz."""

    @staticmethod
    def forward(ctx, x, w):
        ctx.save_for_backward(x, w)
        return _matmul(x, w.detach())

    @staticmethod
    def backward(ctx, dz):
        x, w = ctx.saved_tensors
        B, C = x.shape
        N = w.shape[1]
        dz = dz.to(torch.float32).contiguous()
        dx = _gemm(0, 1, B, C, N, dz, w, torch.empty(B, C, dtype=torch.float32, device=x.device)) if ctx.needs_input_grad[0] else None
        dw = _gemm(1, 0, C, N, B, x, dz, torch.empty(C, N, dtype=torch.float32, device=x.device)) if ctx.needs_input_grad[1] else None
        return dx, dw


def _invconv_compose(p, l, u, log_s, sign_s, reverse):
    """W (and W^-1 when reverse) of one LU-parametrised 1x1 conv (lfi_invconv_compose, K = 1)."""
    C = l.shape[0]
    dev = l.device
    L = cabi.lib()
    w = torch.empty(C, C, dtype=torch.float32, device=dev)
    winv = torch.empty(C, C, dtype=torch.float32, device=dev) if reverse else None
    ws = torch.empty(L.lfi_invconv_ws_bytes(1, C), dtype=torch.uint8, device=dev)
    cabi.check(L.lfi_invconv_compose(1, C, cabi.ptr(p), cabi.ptr(l), cabi.ptr(u), cabi.ptr(log_s), cabi.ptr(sign_s), cabi.ptr(w),
                                     cabi.ptr(winv), ws.data_ptr(), ws.numel(), cabi.stream_ptr()), "lfi_invconv_compose")
    return w, winv


class _InvConvWeightFn(torch.autograd.Function):
    """InvertibleConv1x1.get_weight with LU under autograd (modules.py:163-178): forward = lfi_invconv_compose, backward =
    lfi_invconv_compose_bwd; in the reverse direction dW = -W^-T dW^-1 W^-T first."""

    @staticmethod
    def forward(ctx, l, u, log_s, p, sign_s, reverse):
        w, winv = _invconv_compose(p, l.detach(), u.detach(), log_s.detach(), sign_s, reverse)
        ctx.reverse = reverse
        ctx.save_for_backward(l, u, log_s, p, sign_s, winv)
        return winv if reverse else w

    @staticmethod
    def backward(ctx, dw):
        l, u, log_s, p, sign_s, winv = ctx.saved_tensors
        C = l.shape[0]
        dev = l.device
        dw = dw.to(torch.float32).contiguous()
        if ctx.reverse:  # M = W^-1: dL/dW = -M^T (dL/dM) M^T
            t = _gemm(0, 1, C, C, C, dw, winv, torch.empty(C, C, dtype=torch.float32, device=dev))
            dw = _gemm(1, 0, C, C, C, winv, t, torch.empty(C, C, dtype=torch.float32, device=dev)).neg_()
        L = cabi.lib()
        # lfi_invconv_compose_bwd accumulates, and only into the entries the LU masks keep: the rest stays exactly 0
        dl, du = torch.zeros(C, C, dtype=torch.float32, device=dev), torch.zeros(C, C, dtype=torch.float32, device=dev)
        dls = torch.zeros(C, dtype=torch.float32, device=dev)
        ws = torch.empty(L.lfi_invconv_ws_bytes(1, C), dtype=torch.uint8, device=dev)
        cabi.check(L.lfi_invconv_compose_bwd(1, C, cabi.ptr(p), cabi.ptr(l), cabi.ptr(u), cabi.ptr(log_s), cabi.ptr(sign_s), cabi.ptr(dw),
                                             cabi.ptr(dl), cabi.ptr(du), cabi.ptr(dls), ws.data_ptr(), ws.numel(), cabi.stream_ptr()),
                   "lfi_invconv_compose_bwd")
        return dl, du, dls, None, None, None


def _linear_zeros(x, weight, bias, logs, factor):
    B = x.shape[0]
    out = torch.empty(B, weight.shape[0], dtype=torch.float32, device=x.device)
    cabi.check(cabi.lib().lfi_matmul(cabi.ptr(x), cabi.ptr(weight), cabi.ptr(bias), cabi.ptr(out), B, weight.shape[0], weight.shape[1], 1,
                                     cabi.stream_ptr()), "lfi_matmul")
    return out * torch.exp(logs * factor)


class _LinearZerosFn(torch.autograd.Function):
    """LinearZeros.forward under autograd: the inference launches forward, lfi_linear_zeros_bwd backward."""

    @staticmethod
    def forward(ctx, x, weight, bias, logs, factor):
        out = _linear_zeros(x, weight.detach(), bias.detach(), logs.detach(), factor)
        ctx.factor = factor
        ctx.save_for_backward(x, weight, bias, logs, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, weight, _, logs, out = ctx.saved_tensors
        B, In = x.shape
        Out = weight.shape[0]
        dev = x.device
        dout = dout.to(torch.float32).contiguous()
        dx = torch.empty(B, In, dtype=torch.float32, device=dev)
        dw = torch.empty(Out, In, dtype=torch.float32, device=dev)
        db = torch.empty(Out, dtype=torch.float32, device=dev)
        dlogs = torch.empty(Out, dtype=torch.float32, device=dev)
        L = cabi.lib()
        ws = torch.empty(L.lfi_linear_zeros_bwd_ws_bytes(B, Out), dtype=torch.uint8, device=dev)
        cabi.check(L.lfi_linear_zeros_bwd(cabi.ptr(x), cabi.ptr(weight), cabi.ptr(logs), cabi.ptr(out), cabi.ptr(dout), float(ctx.factor),
                                          cabi.ptr(dx), cabi.ptr(dw), cabi.ptr(db), cabi.ptr(dlogs), B, In, Out, ws.data_ptr(), ws.numel(),
                                          cabi.stream_ptr()), "lfi_linear_zeros_bwd")
        return dx, dw, db, dlogs, None


class ActNorm2d(nn.Module):
    """y = (x + bias) * exp(logs), per channel on [B, C]; log-det term C * sum(logs) (the reference
    multiplies by input.size(1), modules.py:62).  Data-dependent init on the first training call
    (modules.py:32-43)."""

    def __init__(self, num_features, scale=1.0):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(1, num_features))
        self.logs = nn.Parameter(torch.zeros(1, num_features))
        self.num_features = num_features
        self.scale = float(scale)
        self.inited = False

    def initialize_parameters(self, input):
        if not self.training:
            return
        assert input.device == self.bias.device
        with torch.no_grad():
            x = input.detach().float()
            bias = -x.mean(dim=0, keepdim=True)
            var = ((x + bias) ** 2).mean(dim=0, keepdim=True)
            logs = torch.log(self.scale / (torch.sqrt(var) + 1e-6))
            self.bias.data.copy_(bias)
            self.logs.data.copy_(logs)
            self.inited = True

    def forward(self, input, logdet=None, reverse=False):
        if not self.inited:
            self.initialize_parameters(input)
        if _needs_grad(input, self.bias, self.logs):
            x = input.to(torch.float32).contiguous()
            y = _ActNormFn.apply(x, _f32g(self.bias, x.device), _f32g(self.logs, x.device), bool(reverse))
            logs = self.logs
        else:
            x = _f32c(input)
            y = _actnorm(x, _f32c(self.bias, x.device), _f32c(self.logs, x.device), reverse)
            logs = self.logs.detach()
        if logdet is not None:
            dlogdet = logs.sum().to(x.device) * x.shape[1]
            logdet = logdet - dlogdet if reverse else logdet + dlogdet
        return y, logdet


class LinearZeros(nn.Linear):
    """(h W^T + b) * exp(logs * logscale_factor), zero initialised (modules.py:83-95)."""

    def __init__(self, in_channels, out_channels, logscale_factor=3):
        super().__init__(in_channels, out_channels)
        self.logscale_factor = logscale_factor
        self.logs = nn.Parameter(torch.zeros(out_channels))
        self.weight.data.zero_()
        self.bias.data.zero_()

    def forward(self, input):
        if _needs_grad(input, self.weight, self.bias, self.logs):
            x = input.to(torch.float32).contiguous()
            dev = x.device
            return _LinearZerosFn.apply(x, _f32g(self.weight, dev), _f32g(self.bias, dev), _f32g(self.logs, dev), self.logscale_factor)
        x = _f32c(input)
        return _linear_zeros(x, _f32c(self.weight, x.device), _f32c(self.bias, x.device), _f32c(self.logs, x.device), self.logscale_factor)


class InvertibleConv1x1(nn.Module):
    """z = x @ W with W = P (L*mask + I)(U*mask^T + diag(sign_s e^{log_s})) when LU_decomposed
    (modules.py:122-194); log-det term C * sum(log_s).  Init: QR of a numpy Gaussian + scipy LU,
    drawn exactly as the reference draws it (modules.py:126-143)."""

    def __init__(self, num_channels, LU_decomposed=False):
        super().__init__()
        w_shape = [num_channels, num_channels]
        w_init = np.linalg.qr(np.random.randn(*w_shape))[0].astype(np.float32)
        if not LU_decomposed:
            self.weight = nn.Parameter(torch.Tensor(w_init))
        else:
            np_p, np_l, np_u = scipy.linalg.lu(w_init)
            np_s = np.diag(np_u)
            self.register_buffer("p", torch.Tensor(np_p.astype(np.float32)))
            self.register_buffer("sign_s", torch.Tensor(np.sign(np_s).astype(np.float32)))
            self.l = nn.Parameter(torch.Tensor(np_l.astype(np.float32)))
            self.log_s = nn.Parameter(torch.Tensor(np.log(np.abs(np_s)).astype(np.float32)))
            self.u = nn.Parameter(torch.Tensor(np.triu(np_u, k=1).astype(np.float32)))
        self.w_shape = w_shape
        self.LU = LU_decomposed

    def _params(self):
        return [self.l, self.u, self.log_s] if self.LU else [self.weight]

    def get_weight(self, input, reverse):
        """(W, or W^-1 when reverse, and the log-det term C * log|det W|); carries grad to the parameters when grad mode is on
        and one of them requires grad."""
        dev = input.device
        grad = _needs_grad(*self._params())
        if not self.LU:
            w = _f32g(self.weight, dev) if grad else _f32c(self.weight, dev)
            dlogdet = torch.slogdet(w)[1] * input.size(1)
            if reverse:
                w = torch.inverse(w.double()).float()
            return w, dlogdet
        p, sign_s = _f32c(self.p, dev), _f32c(self.sign_s, dev)
        if grad:
            w = _InvConvWeightFn.apply(_f32g(self.l, dev), _f32g(self.u, dev), _f32g(self.log_s, dev), p, sign_s, bool(reverse))
            return w, self.log_s.sum().to(dev) * input.size(1)
        w, winv = _invconv_compose(p, _f32c(self.l, dev), _f32c(self.u, dev), _f32c(self.log_s, dev), sign_s, reverse)
        return (winv if reverse else w), self.log_s.detach().sum().to(dev) * input.size(1)

    def forward(self, input, logdet=None, reverse=False):
        if _needs_grad(input, *self._params()):
            x = input.to(torch.float32).contiguous()
            weight, dlogdet = self.get_weight(x, reverse)
            z = _MatmulFn.apply(x, weight.contiguous())
        else:
            x = _f32c(input)
            weight, dlogdet = self.get_weight(x, reverse)
            z = _matmul(x, weight.contiguous())
        if logdet is not None:
            logdet = logdet - dlogdet if reverse else logdet + dlogdet
        return z, logdet


class GaussianDiag:
    """Standard-normal prior helpers (modules.py:197-235)."""

    Log2PI = float(np.log(2 * np.pi))

    @staticmethod
    def likelihood_simplified(x):
        return -0.5 * ((x ** 2) + GaussianDiag.Log2PI)

    @staticmethod
    def logp_simplified(x):
        return torch.sum(GaussianDiag.likelihood_simplified(x), dim=1)

    @staticmethod
    def likelihood(mean, logs, x):
        return -0.5 * (logs * 2.0 + ((x - mean) ** 2) / torch.exp(logs * 2.0) + GaussianDiag.Log2PI)

    @staticmethod
    def logp(mean, logs, x):
        return torch.sum(GaussianDiag.likelihood(mean, logs, x), dim=1)

    @staticmethod
    def sample(output_shape, eps_std=1):
        return torch.normal(mean=torch.zeros_like(output_shape), std=torch.ones_like(output_shape) * eps_std)

    @staticmethod
    def nll_bits(z, logdet):
        """-(logdet + logp_simplified(z)) / ln 2 on the device (SeqGlow.loss, models.py:563-565)."""
        z = _f32c(z)
        ld = _f32c(logdet)
        out = torch.empty(z.shape[0], dtype=torch.float32, device=z.device)
        cabi.check(cabi.lib().lfi_nll(cabi.ptr(z), cabi.ptr(ld), cabi.ptr(out), z.shape[0], z.shape[1], cabi.stream_ptr()), "lfi_nll")
        return out
