"""Conditional Glow (MoGlow-style) with the reference's module API, backed by the sm_100a kernels.

Class names, constructor signatures, parameter names/shapes and the `forward` conventions follow
`code/glow_pytorch/glow/models.py` of the reference (file:line cited per class) so this package is
a drop-in for `glow_pytorch.glow`; the per-frame Python loops of the reference are replaced by
three fused device paths reached through the C ABI (`engine.py` / `_cabi.py`):

  SeqGlow.forward   -> lfi_seq_train_fwd / lfi_seq_train_bwd  (autograd.Function below; lfi_seq_train_bwd_dx when a batch
                       stream requires grad)
  SeqGlow.inference -> lfi_seq_sample (persistent autoregressive sampler)
  SeqGlow.invert    -> lfi_seq_sample (teacher forced)
  FlowStep / FlowNet / Glow single-frame calls -> lfi_flowstep (under autograd lfi_flowstep_fwd_train / lfi_flowstep_bwd, in the
                                                  reverse direction lfi_flowstep_rev_fwd_train / lfi_flowstep_rev_bwd)
  f_seq.forward on its own                     -> lfi_fseq_fwd (under autograd lfi_fseq_bwd as well)

CUDA tensors only; there is no CPU / eager fallback.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _cabi as cabi
from ..engine import MODALITIES, Engine, feature_train_bwd, feature_train_fwd
from . import modules, thops
from .modules import GaussianDiag
from .utils import get_longest_history

LN2 = float(np.log(2.0))


class ModalityEncoder(nn.Module):
    """One conditioning stream (reference models.py:12-80).  `enc: rnn` (1-layer batch-first GRU from a
    zero state, output = final state twice) and `enc: none` (flattened window) run on the device path;
    the lstm / mlp / cnn variants are constructed (so the RNG stream and state-dict match) but are outside
    the accelerated path (SURVEY.md §2 row 5)."""

    def __init__(self, input_size, params):
        super().__init__()
        self.dropout = nn.Dropout(params["dropout"]) if params["dropout"] > 0 else None
        self.input_size = input_size
        self.history = params["history"]
        self.enc_type = params["enc"]
        if params["enc"] == "rnn":
            self.encoder = nn.GRU(input_size=input_size, hidden_size=params["hidden_dim"], batch_first=True)
            self.dim = params["hidden_dim"] * 2
        elif params["enc"] == "lstm":
            self.encoder = nn.LSTM(input_size=input_size, hidden_size=params["hidden_dim"], batch_first=True)
            self.dim = params["hidden_dim"] * 2
        elif params["enc"] == "mlp":
            self.encoder = nn.Sequential(nn.Linear(input_size * params["history"], params["hidden_dim"]), nn.LeakyReLU())
            self.dim = params["hidden_dim"]
        elif params["enc"] == "cnn":
            self.encoder = nn.Conv1d(input_size, params["hidden_dim"], params["kernel_size"], padding=params["kernel_size"] // 2)
            self.dim = input_size - params["kernel_size"] + 1
        elif params["enc"] == "none":
            self.encoder = None
            self.dim = input_size * params["history"]
        else:
            raise NotImplementedError()

    def draw_mask(self, lead_shape, device):
        """Frame-dropout mask as the reference draws it: Dropout(p)(ones[..., hist]) (models.py:56-58)."""
        if not (self.training and self.dropout is not None):
            return None
        return self.dropout(torch.ones(*lead_shape, self.history, device=device))

    def forward(self, x):
        """x: [B, hist, d] -> [B, dim].  Runs the window through the device encoder path."""
        if self.enc_type not in ("rnn", "none"):
            raise NotImplementedError("enc=%r is outside the accelerated path" % self.enc_type)
        fe = _SingleModality(self)
        mask = self.draw_mask(x.shape[:1], x.device)
        params = fe.gru_params()
        if modules._needs_grad(x, *params):
            return fe.encode_autograd(x, mask, params)
        return fe.encode(x, mask)


class FeatureEncoder(nn.Module):
    """Concatenates the modality encodings in the order p1_face | p2_face | p1_speech | p2_speech
    (reference models.py:83-145)."""

    def __init__(self, conditioning_hparams, data_hparams):
        super().__init__()
        self.use_frame_nb = conditioning_hparams["use_frame_nb"]
        self.p1_speech_history = conditioning_hparams["p1_speech"]["history"]
        self.p2_speech_history = conditioning_hparams["p2_speech"]["history"]
        self.p2_face_history = conditioning_hparams["p2_face"]["history"]
        speech_dim = data_hparams["speech_dim"]
        self._in_dim = {"p1_face": conditioning_hparams["p1_face"]["dim"], "p2_face": conditioning_hparams["p2_face"].get("dim", 0),
                        "p1_speech": speech_dim, "p2_speech": speech_dim}
        self._hist = {m: conditioning_hparams[m]["history"] for m in MODALITIES}

        self.p1_face_encoder = ModalityEncoder(conditioning_hparams["p1_face"]["dim"], conditioning_hparams["p1_face"])
        self.dim = self.p1_face_encoder.dim
        if self.p2_face_history:
            self.p2_face_encoder = ModalityEncoder(conditioning_hparams["p2_face"]["dim"], conditioning_hparams["p2_face"])
            self.dim += self.p2_face_encoder.dim
        if self.p1_speech_history:
            self.p1_speech_encoder = ModalityEncoder(speech_dim, conditioning_hparams["p1_speech"])
            self.dim += self.p1_speech_encoder.dim
        if self.p2_speech_history:
            self.p2_speech_encoder = ModalityEncoder(speech_dim, conditioning_hparams["p2_speech"])
            self.dim += self.p2_speech_encoder.dim
        if self.use_frame_nb:
            self.dim += 1
        self._engine = None

    # -- facts the engine needs ------------------------------------------------------------
    def encoder_of(self, m):
        return getattr(self, m + "_encoder", None) if (m == "p1_face" or self._hist[m]) else None

    def modality_info(self, m):
        """(history, raw dim, GRU hidden or 0) for lfi_shape; unsupported encoders raise."""
        enc = self.encoder_of(m)
        if enc is None:
            return 0, 0, 0
        if self.use_frame_nb:
            raise NotImplementedError("use_frame_nb is outside the accelerated path (false in every shipped yaml)")
        if enc.enc_type == "rnn":
            return self._hist[m], self._in_dim[m], enc.encoder.hidden_size
        if enc.enc_type == "none":
            return self._hist[m], self._in_dim[m], 0
        raise NotImplementedError("enc=%r is outside the accelerated path (SURVEY.md §2 row 5)" % enc.enc_type)

    def gru_of(self, m):
        enc = self.encoder_of(m)
        return enc.encoder if (enc is not None and enc.enc_type == "rnn") else None

    def draw_masks(self, lead_shape, device):
        out = {}
        for m in MODALITIES:
            enc = self.encoder_of(m)
            out[m] = enc.draw_mask(lead_shape, device) if enc is not None else None
        return out if any(v is not None for v in out.values()) else None

    def gru_params(self):
        """The GRU parameters of every GRU-encoded modality, MODALITIES order, (weight_ih, weight_hh, bias_ih, bias_hh) each."""
        out = []
        for m in MODALITIES:
            gru = self.gru_of(m)
            if gru is not None:
                out += [gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0]
        return out

    def forward(self, condition):
        """condition: {"prev_p1_face": [B,h0,C], "p2_face": [B,h,d], "p1_speech": ..., "p2_speech": ...} -> [B, dim].
        With grad mode on and a window or a GRU parameter requiring grad, the call is one autograd node (_FeatureEncodeFn)."""
        eng = self._engine if self._engine is not None else _encoder_only_engine(self)
        x0 = condition["prev_p1_face"]
        B, dev = x0.shape[0], x0.device
        st = eng.start_ts
        wins, data = {}, {}
        for m in MODALITIES:
            h = self._hist[m]
            if m != "p1_face" and not h:
                continue
            win = condition["prev_p1_face" if m == "p1_face" else m]
            wins[m] = win
            buf = torch.zeros(B, st + 1, win.shape[2], device=dev)
            if m == "p1_face":
                buf[:, st - h:st] = win.float()      # window [t-h, t)
            else:
                buf[:, st - h + 1:st + 1] = win.float()  # window (t-h, t]
            data[m] = buf
        masks = self.draw_masks((1, B), dev)
        params = self.gru_params()
        if not modules._needs_grad(*wins.values(), *params):
            return eng.unfold_features(eng.feature_encode(data, st, 1, masks))
        # the window gradients leave the node as gradients of the padded buffers; the slice assignments above carry them back
        bufs = [data.get(m) for m in MODALITIES]

        def fwd(bs):
            return eng.feature_encode_train({m: b for m, b in zip(MODALITIES, bs) if b is not None}, st, 1, masks)

        cond = _FeatureEncodeFn.apply(fwd, eng.feature_encode_backward, len(bufs), *bufs, *params)
        return eng.unfold_features(cond)


def _encoder_only_engine(fe):
    eng = Engine([], fe)
    fe._engine = eng
    eng.ensure()
    return eng


class _FeatureEncodeFn(torch.autograd.Function):
    """The window encoders under autograd (reference models.py:55-80 differentiated by torch): forward = `fwd(bufs)` over
    lfi_feature_encode_fwd_train, backward = `bwd(saved, dcond, want_dx)` over lfi_feature_encode_bwd.  Inputs after `n` are
    the n padded stream buffers [B, T, dim] (MODALITIES order, None where absent) and then the GRU parameters in
    `FeatureEncoder.gru_params()` order (graph connectivity; the calls read the values through their own pointers).  The node
    keeps its stash and masks; the backward runs in the forward's gemm mode."""

    @staticmethod
    def forward(ctx, fwd, bwd, n, *tensors):
        cond, saved = fwd(tensors[:n])
        ctx.bwd, ctx.saved, ctx.n = bwd, saved, n
        return cond

    @staticmethod
    def backward(ctx, dcond):
        n = ctx.n
        want = ctx.needs_input_grad[3:3 + n]
        dx, grads = ctx.bwd(ctx.saved, dcond, want)
        dparams = [g for gs in grads if gs is not None for g in gs]
        return (None, None, None) + tuple(dx[:n]) + tuple(dparams)


class _SingleModality:
    """Runs one ModalityEncoder window through lfi_feature_encode (a p1_face dummy fills slot 0), under autograd through
    lfi_feature_encode_fwd_train / lfi_feature_encode_bwd."""

    def __init__(self, enc: ModalityEncoder):
        self.enc = enc

    def gru_params(self):
        g = self.enc.encoder if self.enc.enc_type == "rnn" else None
        return [g.weight_ih_l0, g.weight_hh_l0, g.bias_ih_l0, g.bias_hh_l0] if g is not None else []

    def _call(self, xb, mask, params):
        """Shape, Params and Batch of the one-modality call: xb [B, h+1, d] = the window after one zero frame (slot 1), params fp32
        on xb's device."""
        enc = self.enc
        B, T, d = xb.shape
        h = T - 1
        dev = xb.device
        sh = cabi.Shape()
        sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps, sh.f_raw = 2, 1, 4, 4, 3, 1, 1e-4, 0
        sh.hist[0], sh.dim[0], sh.ehid[0] = 1, 2, 0
        E = enc.encoder.hidden_size if enc.enc_type == "rnn" else 0
        sh.hist[1], sh.dim[1], sh.ehid[1] = h, d, E
        P = cabi.Params()
        keep = list(params)
        for name, t in zip(("enc_w_ih", "enc_w_hh", "enc_b_ih", "enc_b_hh"), params):
            getattr(P, name)[1] = cabi.ptr(t)
        bt = cabi.Batch()
        bt.B, bt.T = B, T
        dummy = torch.zeros(B, T, 2, device=dev)
        keep += [dummy, xb]
        bt.x[0], bt.x[1] = cabi.ptr(dummy), cabi.ptr(xb)
        if mask is not None:
            mk = mask.reshape(1, B, h).float().contiguous()
            keep.append(mk)
            bt.mask[1] = cabi.ptr(mk)
        return sh, P, bt, keep

    def encode_autograd(self, x, mask, params):
        B, h, d = x.shape
        dev = x.device
        xb = torch.zeros(B, h + 1, d, device=dev)
        xb[:, 1:] = x.float()
        params = [modules._f32g(p, dev) for p in params]

        def fwd(bs):
            sh, P, bt, keep = self._call(bs[1].detach(), mask, [p.detach() for p in params])
            return feature_train_fwd(sh, P, bt, keep, h, 1, cabi.GEMM_FP32, dev)

        cond = _FeatureEncodeFn.apply(fwd, feature_train_bwd, 2, None, xb, *params)
        out = cond[:, 2:]
        return torch.cat([out, out], dim=1) if params else out

    def encode(self, x, mask):
        import ctypes
        B, h, d = x.shape
        dev = x.device
        E = self.enc.encoder.hidden_size if self.enc.enc_type == "rnn" else 0
        xb = torch.zeros(B, h + 1, d, device=dev)
        xb[:, 1:] = x.float()
        sh, P, bt, keep = self._call(xb, mask, [modules._f32c(p, dev) for p in self.gru_params()])
        T = h + 1
        L = cabi.lib()
        Fe = L.lfi_feature_dim_folded(ctypes.byref(sh))
        cond = torch.empty(B, Fe, device=dev)
        ws = torch.empty(L.lfi_feature_ws_bytes(ctypes.byref(sh), B, T, 1, cabi.GEMM_FP32), dtype=torch.uint8, device=dev)
        cabi.check(L.lfi_feature_encode(ctypes.byref(sh), ctypes.byref(P), ctypes.byref(bt), h, 1, cabi.ptr(cond), ws.data_ptr(),
                                        ws.numel(), cabi.GEMM_FP32, cabi.stream_ptr()), "lfi_feature_encode")
        out = cond[:, 2:]
        return torch.cat([out, out], dim=1) if E else out


def _fseq_run(shape, params, z, cond, h_in, c_in, want_stash):
    """lfi_fseq_fwd on device tensors (fp32, contiguous): returns (out, h, c or None, stash or None)."""
    L = cabi.lib()
    B, dev = z.shape[0], z.device
    h = torch.empty(B, shape.H, dtype=torch.float32, device=dev)
    c = torch.empty(B, shape.H, dtype=torch.float32, device=dev) if shape.G == 4 else None
    out = torch.empty(B, shape.Out, dtype=torch.float32, device=dev)
    stash = torch.empty(L.lfi_fseq_stash_bytes(ctypes.byref(shape), B), dtype=torch.uint8, device=dev) if want_stash else None
    ws = torch.empty(L.lfi_fseq_ws_bytes(ctypes.byref(shape), B), dtype=torch.uint8, device=dev)
    P = cabi.FseqParams(*[cabi.ptr(t) for t in params])
    cabi.check(L.lfi_fseq_fwd(ctypes.byref(shape), ctypes.byref(P), cabi.ptr(z), cabi.ptr(cond), cabi.ptr(h_in), cabi.ptr(c_in), cabi.ptr(h),
                              cabi.ptr(c), cabi.ptr(out), B, stash.data_ptr() if want_stash else None, stash.numel() if want_stash else 0, ws.data_ptr(),
                              ws.numel(), cabi.stream_ptr()), "lfi_fseq_fwd")
    return out, h, c, stash


class _FSeqFn(torch.autograd.Function):
    """f_seq.forward under autograd (reference models.py:204-214 differentiated by torch): forward = lfi_fseq_fwd with a stash,
    backward = lfi_fseq_bwd.  Inputs after `c_in` are the nine parameters in `f_seq._params()` order."""

    @staticmethod
    def forward(ctx, shape, z, cond, h_in, c_in, *params):
        out, h, c, stash = _fseq_run(shape, [p.detach() for p in params], z.detach(), cond.detach(),
                                     h_in.detach() if h_in is not None else None, c_in.detach() if c_in is not None else None, True)
        ctx.shape, ctx.stash = shape, stash
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(z, cond, h_in, c_in, *params)
        return (out, h) + ((c,) if c is not None else ())

    @staticmethod
    def backward(ctx, dout, dh, dc=None):
        shape, stash = ctx.shape, ctx.stash
        z, cond, h_in, c_in, *params = ctx.saved_tensors
        B, dev = z.shape[0], z.device
        f32 = lambda t: t.to(dtype=torch.float32).contiguous() if t is not None else None
        dout = f32(dout) if dout is not None else torch.zeros(B, shape.Out, dtype=torch.float32, device=dev)
        dh, dc = f32(dh), f32(dc)
        dz, dcond = torch.empty_like(z), torch.empty_like(cond)
        dh_in = torch.empty_like(h_in) if h_in is not None else None
        dc_in = torch.empty_like(c_in) if c_in is not None else None
        grads = [torch.empty_like(p) for p in params]
        L = cabi.lib()
        ws = torch.empty(L.lfi_fseq_bwd_ws_bytes(ctypes.byref(shape), B), dtype=torch.uint8, device=dev)
        P = cabi.FseqParams(*[cabi.ptr(t) for t in params])
        Gr = cabi.FseqParams(*[cabi.ptr(t) for t in grads])
        cabi.check(L.lfi_fseq_bwd(ctypes.byref(shape), ctypes.byref(P), cabi.ptr(z), cabi.ptr(cond), cabi.ptr(h_in), cabi.ptr(c_in),
                                  cabi.ptr(dout), cabi.ptr(dh), cabi.ptr(dc), cabi.ptr(dz), cabi.ptr(dcond), cabi.ptr(dh_in), cabi.ptr(dc_in),
                                  ctypes.byref(Gr), B, stash.data_ptr(), stash.numel(), ws.data_ptr(), ws.numel(), cabi.stream_ptr()),
                   "lfi_fseq_bwd")
        return (None, dz, dcond, dh_in, dc_in) + tuple(grads)


class f_seq(nn.Module):
    """Coupling network: Linear+LeakyReLU on the conditioning, GRUCell/LSTMCell over frames, LinearZeros
    (reference models.py:148-214).  Holds the parameters and the carried RNN state.  Inside a FlowStep it is evaluated by the
    fused flow-step kernels; `forward` runs it on its own (lfi_fseq_fwd, under autograd lfi_fseq_bwd as well) and leaves the
    state where FlowStep.forward of the same step reads it next."""

    def __init__(self, input_size, output_size, hidden_size, cond_dim, feature_encoder_dim, rnn_type):
        super().__init__()
        self.hidden_size = hidden_size
        self.input_size = input_size
        self.output_size = output_size
        self.rnn_type = rnn_type
        if rnn_type == "gru":
            self.rnn = nn.GRUCell(input_size=input_size + cond_dim, hidden_size=hidden_size)
        elif rnn_type == "lstm":
            self.rnn = nn.LSTMCell(input_size=input_size + cond_dim, hidden_size=hidden_size)
        else:
            raise NotImplementedError("rnn_type must be 'gru' or 'lstm'")
        self.cond_transform = nn.Sequential(nn.Linear(feature_encoder_dim, cond_dim), nn.LeakyReLU())
        self.final_linear = modules.LinearZeros(hidden_size, output_size)
        self.hidden = None
        self.cell = None

    def init_rnn_hidden(self):
        """None == zero state (models.py:196-202)."""
        self.hidden = None
        self.cell = None

    def _params(self):
        ct, fl = self.cond_transform[0], self.final_linear
        return [ct.weight, ct.bias, self.rnn.weight_ih, self.rnn.bias_ih, self.rnn.weight_hh, self.rnn.bias_hh, fl.weight, fl.bias, fl.logs]

    def _shape(self):
        sh = cabi.FseqShape()
        ct = self.cond_transform[0]
        sh.In, sh.Out, sh.H, sh.D, sh.F = self.input_size, self.output_size, self.hidden_size, ct.out_features, ct.in_features
        sh.G = 3 if self.rnn_type == "gru" else 4
        sh.logscale_factor = float(self.final_linear.logscale_factor)
        return sh

    def forward(self, z, condition):
        """z [B, input_size], condition [B, feature_encoder_dim] -> [B, output_size]; updates self.hidden (and self.cell)."""
        params = self._params()
        h_in, c_in = self.hidden, (self.cell if self.rnn_type == "lstm" else None)
        dev = z.device
        sh = self._shape()
        B = z.shape[0]
        if z.shape[1] != sh.In or condition.shape != (B, sh.F):
            raise RuntimeError("f_seq expects z [B,%d] and condition [B,%d], got %s / %s" % (sh.In, sh.F, tuple(z.shape), tuple(condition.shape)))
        for name, t in (("hidden", h_in), ("cell", c_in)):
            if t is not None and t.shape != (B, sh.H):
                raise RuntimeError("f_seq.%s has shape %s, expected [%d, %d]" % (name, tuple(t.shape), B, sh.H))
        if modules._needs_grad(z, condition, h_in, c_in, *params):
            f32 = lambda t: modules._f32g(t, dev) if t is not None else None
            outs = _FSeqFn.apply(sh, f32(z), f32(condition), f32(h_in), f32(c_in), *[f32(p) for p in params])
            out, h, c = outs[0], outs[1], (outs[2] if sh.G == 4 else None)
        else:
            f32 = lambda t: modules._f32c(t, dev) if t is not None else None
            out, h, c, _ = _fseq_run(sh, [f32(p) for p in params], f32(z), f32(condition), f32(h_in), f32(c_in), False)
        self.hidden, self.cell = h, c
        return out


class _FlowStepFn(torch.autograd.Function):
    """One FlowStep on one frame under autograd (reference: FlowStep.normal_flow, models.py:311-342, or with reverse set
    FlowStep.reverse_flow, models.py:345-373, differentiated by torch): forward = lfi_flowstep_fwd_train / lfi_flowstep_rev_fwd_train,
    backward = lfi_flowstep_bwd / lfi_flowstep_rev_bwd + the LU chain rule.  Inputs after `c_in` are the step's parameters in
    `FlowStep._autograd_params()` order (graph connectivity; values are read from the flat buffer).  The reverse node also saves
    them, so that an in-place update between its forward and backward raises instead of differentiating the wrong W^-1."""

    @staticmethod
    def forward(ctx, eng, k, want_scale, n_lu, refresh, reverse, x, cond, h_in, c_in, *params):
        y, ld, h_out, c_out, scale, saved = eng.flowstep_train(k, x, cond, h_in, c_in, want_scale, refresh=refresh, reverse=reverse)
        ctx.eng, ctx.k, ctx.saved, ctx.n_lu, ctx.reverse = eng, k, saved, n_lu, reverse
        if reverse:
            ctx.save_for_backward(*params)
        ctx.has_c = c_out is not None
        outs = (y, ld, h_out) + ((c_out,) if c_out is not None else ()) + ((scale,) if scale is not None else ())
        if scale is not None:
            ctx.mark_non_differentiable(scale)
        ctx.n_out = len(outs)
        return outs

    @staticmethod
    def backward(ctx, *grads):
        eng, k = ctx.eng, ctx.k
        dy, dld, dh_out = grads[0], grads[1], grads[2]
        dc_out = grads[3] if ctx.has_c else None
        if ctx.reverse:
            ctx.saved_tensors  # raises if a parameter changed in place since the forward
        dx, dcond, dh_in, dc_in, g = eng.flowstep_backward(k, ctx.saved, dy, dld, dh_out, dc_out, reverse=ctx.reverse)
        C = eng.C
        out = [g["an_bias"].view(1, C), g["an_logs"].view(1, C)]
        if ctx.n_lu:
            dl, du, dls = eng.invconv_chain_rule(k, g["w"])
            out += [dl, du, dls]
        else:
            out += [g["w"].view(C, C)]
        GH, In, H, D, F, Co = eng.G * eng.H, eng.Ci + eng.D, eng.H, eng.D, eng.F, eng.Co
        out += [g["wc"].view(D, F), g["bc"], g["w_ih"].view(GH, In), g["b_ih"], g["w_hh"].view(GH, H), g["b_hh"],
                g["wf"].view(Co, H), g["bf"], g["lf"]]
        _, h_in, c_in = ctx.saved[1], ctx.saved[2], ctx.saved[3]
        return (None, None, None, None, None, None, dx, dcond, dh_in if h_in is not None else None,
                dc_in if (c_in is not None and dc_in is not None) else None) + tuple(out)


class FlowStep(nn.Module):
    """ActNorm -> invertible 1x1 conv -> affine/additive coupling (reference models.py:217-376)."""

    FlowCoupling = ["additive", "affine"]
    FlowPermutation = ["reverse", "shuffle", "invconv"]

    def __init__(self, in_channels, hidden_channels, cond_dim, actnorm_scale=1.0, flow_permutation="shuffle",
                 flow_coupling="additive", LU_decomposed=False, L=1, K=1, scale_eps=1e-6, scale_logging=False,
                 feature_encoder_dim=0, glow_rnn_type=None):
        assert flow_coupling in FlowStep.FlowCoupling, "flow_coupling should be in `{}`".format(FlowStep.FlowCoupling)
        assert flow_permutation in FlowStep.FlowPermutation, "float_permutation should be in `{}`".format(FlowStep.FlowPermutation)
        super().__init__()
        if flow_permutation != "invconv":
            raise NotImplementedError("only flow_permutation='invconv' is live in the reference (Permute2d asserts 4-D input and "
                                      "uses np.long, modules.py:98-119)")
        self.flow_permutation = flow_permutation
        self.flow_coupling = flow_coupling
        self.scale = None
        self.scale_logging = scale_logging
        self.scale_eps = scale_eps
        self.L = L
        self.K = K
        self.actnorm = modules.ActNorm2d(in_channels, actnorm_scale)
        self.invconv = modules.InvertibleConv1x1(in_channels, LU_decomposed=LU_decomposed)
        out = in_channels - in_channels // 2
        if flow_coupling == "affine":
            out = in_channels if in_channels % 2 == 0 else in_channels + 1
        self.f = f_seq(in_channels // 2, out, hidden_channels, cond_dim, feature_encoder_dim, glow_rnn_type)
        self._engine = None
        self._k = 0

    def _eng(self):
        if self._engine is None:
            Engine([self], None)  # registers itself on the step
        return self._engine

    def _autograd_params(self):
        inv = [self.invconv.l, self.invconv.u, self.invconv.log_s] if self.invconv.LU else [self.invconv.weight]
        f = self.f
        return [self.actnorm.bias, self.actnorm.logs] + inv + [f.cond_transform[0].weight, f.cond_transform[0].bias, f.rnn.weight_ih, f.rnn.bias_ih,
                                                              f.rnn.weight_hh, f.rnn.bias_hh, f.final_linear.weight, f.final_linear.bias,
                                                              f.final_linear.logs]

    def _forward_autograd(self, eng, input_, cond, logdet, refresh=True, reverse=False):
        """normal_flow (reverse_flow) under autograd: kernels for everything data dependent, torch for the parameter-only log-det
        terms C * sum(logs) + C * sum(log_s) (modules.py:62, 171) so that autograd owns their gradients.  refresh=False: the caller
        (FlowNet.encode / decode) has rebuilt the derived cache for this call already."""
        params = self._autograd_params()
        h_in, c_in = self.f.hidden, self.f.cell
        outs = _FlowStepFn.apply(eng, self._k, bool(self.scale_logging) and not reverse, 1 if self.invconv.LU else 0, bool(refresh),
                                 bool(reverse), input_, cond, h_in, c_in, *params)
        y, ld, h = outs[0], outs[1], outs[2]
        i = 3
        c = None
        if eng.G == 4:
            c = outs[i]
            i += 1
        if self.scale_logging and eng.affine and not reverse:
            self.scale = outs[i]
        self.f.hidden, self.f.cell = h, c
        C = float(eng.C)
        if reverse:  # the terms of Engine.step_logdet_const, in its order, so that the values are those of the no-grad call
            s = self.actnorm.logs.sum() + (self.invconv.log_s.sum() if self.invconv.LU else torch.slogdet(self.invconv.weight)[1])
            if logdet is not None:
                logdet = logdet + (ld - s * C)
            return y, logdet
        const = self.actnorm.logs.sum() * C
        const = const + (self.invconv.log_s.sum() * C if self.invconv.LU else torch.slogdet(self.invconv.weight)[1] * C)
        if logdet is not None:
            logdet = logdet + ld + const
        return y, logdet

    def forward(self, input_, audio_features, logdet=None, reverse=False, _refresh=True):
        assert audio_features is not None
        eng = self._eng()
        eng.ensure(input_.device if input_.is_cuda else None)
        if not reverse and not self.actnorm.inited:
            self.actnorm.initialize_parameters(input_)
        if not reverse and torch.is_grad_enabled() and (
                input_.requires_grad or audio_features.requires_grad or any(p.requires_grad for p in self._autograd_params())
                or (self.f.hidden is not None and self.f.hidden.requires_grad)):
            return self._forward_autograd(eng, input_, audio_features, logdet, _refresh)
        if reverse and modules._needs_grad(input_, audio_features, self.f.hidden, self.f.cell, *self._autograd_params()):
            return self._forward_autograd(eng, input_, audio_features, logdet, _refresh, reverse=True)
        y, logdet, h, c, scale = eng.flowstep(self._k, input_, audio_features, self.f.hidden, self.f.cell, logdet, bool(reverse),
                                              want_scale=self.scale_logging, refresh=_refresh)
        self.f.hidden, self.f.cell = h, c
        if scale is not None:
            self.scale = scale
        return y, logdet

    def normal_flow(self, input_, condition, logdet):
        return self.forward(input_, condition, logdet, False)

    def reverse_flow(self, input_, condition, logdet):
        return self.forward(input_, condition, logdet, True)

    def init_rnn_hidden(self):
        self.f.init_rnn_hidden()


class FlowNet(nn.Module):
    """K*L flow steps (reference models.py:379-467)."""

    def __init__(self, C, hidden_channels, cond_dim, K, L, actnorm_scale=1.0, flow_permutation="invconv",
                 flow_coupling="additive", LU_decomposed=False, scale_eps=1e-6, scale_logging=False, feature_encoder_dim=0,
                 glow_rnn_type=None):
        super().__init__()
        self.layers = nn.ModuleList()
        self.output_shapes = []
        self.K = K
        self.L = L
        for l in range(L):
            for k in range(K):
                self.layers.append(FlowStep(in_channels=C, hidden_channels=hidden_channels, cond_dim=cond_dim,
                                            actnorm_scale=actnorm_scale, flow_permutation=flow_permutation,
                                            flow_coupling=flow_coupling, LU_decomposed=LU_decomposed, L=l, K=k,
                                            scale_eps=scale_eps, scale_logging=scale_logging,
                                            feature_encoder_dim=feature_encoder_dim, glow_rnn_type=glow_rnn_type))
                self.output_shapes.append([-1, C])
        self._engine = None

    def _eng(self):
        if self._engine is None:
            self._engine = Engine(list(self.layers), None)
        return self._engine

    def forward(self, input_, condition, logdet=0.0, reverse=False, eps_std=None):
        return self.decode(input_, condition, eps_std) if reverse else self.encode(input_, condition, logdet)

    def encode(self, z, condition, logdet=0.0):
        eng = self._eng()
        eng.ensure(z.device if z.is_cuda else None)
        eng.refresh(False)
        for layer in self.layers:
            z, logdet = layer(z, condition, logdet, reverse=False, _refresh=False)
        return z, logdet

    def decode(self, z, condition, eps_std=None):
        eng = self._eng()
        eng.ensure(z.device if z.is_cuda else None)
        eng.refresh(True)
        logdet = 0.0
        for layer in reversed(self.layers):
            z, logdet = layer(z, condition, logdet, reverse=True, _refresh=False)
        return z, logdet

    def init_rnn_hidden(self):
        for layer in self.layers:
            layer.init_rnn_hidden()


class Glow(nn.Module):
    """The flow with its prior (reference models.py:470-521)."""

    def __init__(self, hparams, feature_encoder_dim=0):
        super().__init__()
        self.flow = FlowNet(C=hparams.Conditioning["p1_face"]["dim"], hidden_channels=hparams.Glow["hidden_channels"],
                            cond_dim=hparams.Conditioning["cond_dim"], K=hparams.Glow["K"], L=hparams.Glow["L"],
                            actnorm_scale=hparams.Glow["actnorm_scale"], flow_permutation=hparams.Glow["flow_permutation"],
                            flow_coupling=hparams.Glow["flow_coupling"], LU_decomposed=hparams.Glow["LU_decomposed"],
                            scale_eps=hparams.Glow["scale_eps"], scale_logging=hparams.Validation["scale_logging"],
                            feature_encoder_dim=feature_encoder_dim, glow_rnn_type=hparams.Glow.get("rnn_type") or "gru")

    def forward(self, x=None, condition=None, z=None, eps_std=None, reverse=False, output_shape=None):
        if not reverse:
            return self.normal_flow(x, condition)
        return self.reverse_flow(z, condition, eps_std, output_shape)

    def normal_flow(self, x, condition):
        logdet = torch.zeros_like(x[:, 0])
        return self.flow(x, condition, logdet=logdet, reverse=False)

    def reverse_flow(self, z, condition, eps_std, output_shape):
        with torch.no_grad():
            if z is None:
                z = modules.GaussianDiag.sample(output_shape, eps_std)
            x, logdet = self.flow(z, condition, eps_std=eps_std, reverse=True)
        return x, logdet

    def set_actnorm_init(self, inited=True):
        for name, m in self.named_modules():
            if m.__class__.__name__.find("ActNorm") >= 0:
                m.inited = inited

    def init_rnn_hidden(self):
        self.flow.init_rnn_hidden()


class _SeqGlowFn(torch.autograd.Function):
    """z, nll = SeqGlow core.  `mods` lists the modalities (indices into MODALITIES) whose streams follow it as inputs, each
    the [B, T, dim] fp32 device tensor that `batch` holds for it: their gradients come from lfi_seq_train_bwd_dx.  The remaining
    inputs are the engine's parameters (for graph connectivity; their values are read from the flat buffer they alias)."""

    @staticmethod
    def forward(ctx, eng, batch, masks, scale_out, mods, *inputs):
        z, nll = eng.train_forward(batch, masks, scale_out)
        nll = nll - eng.logdet_const().detach() / LN2
        ctx.eng, ctx.token, ctx.mods = eng, eng._fwd_token, mods
        ctx.T = batch["p1_face"].shape[1]
        ctx.save_for_backward(z)
        ctx.mark_non_differentiable(z)
        return z, nll

    @staticmethod
    def backward(ctx, dz, dnll):
        eng = ctx.eng
        (z,) = ctx.saved_tensors
        g = eng.new_flat_grad()
        if not ctx.mods:
            eng.train_backward(z, dnll, g, ctx.token)
            return (None, None, None, None, None) + tuple(eng.grad_views(g))
        B = z.shape[1]
        dx = [None] * cabi.NMOD
        for i in ctx.mods:
            dx[i] = torch.empty(B, ctx.T, eng.shape.dim[i], dtype=torch.float32, device=z.device)
        eng.train_backward(z, dnll, g, ctx.token, dx=dx)
        return (None, None, None, None, None) + tuple(dx[i] for i in ctx.mods) + tuple(eng.grad_views(g))


class SeqGlow(nn.Module):
    """Sequence driver (reference models.py:524-645)."""

    def __init__(self, hparams) -> None:
        super().__init__()
        self.hparams = hparams
        self.feature_encoder = FeatureEncoder(self.hparams.Conditioning, self.hparams.Data)
        self.glow = Glow(hparams, self.feature_encoder.dim)
        self._engine = None
        self.gemm_mode = cabi.GEMM_FP32
        self.injected_masks = None  # tests: {modality: [T',B,hist]} replaces the drawn dropout masks

    # -- engine -------------------------------------------------------------------------------
    def engine(self) -> Engine:
        if self._engine is None:
            self._engine = Engine(list(self.glow.flow.layers), self.feature_encoder, self.gemm_mode)
            self.glow.flow._engine = self._engine
            self.feature_encoder._engine = self._engine
        self._engine.gemm_mode = self.gemm_mode
        self._engine.ensure()
        return self._engine

    def _masks(self, Tp, B, device):
        if self.injected_masks is not None:
            return self.injected_masks
        if not self.training:
            return None
        return self.feature_encoder.draw_masks((Tp, B), device)

    def _ddi(self, eng, batch, masks):
        """ActNorm data-dependent init on the first training frame, layer by layer (modules.py:32-43 via
        models.py:546-552)."""
        st = eng.start_ts
        m0 = {m: (v[:1].contiguous() if v is not None else None) for m, v in masks.items()} if masks else None
        with torch.no_grad():
            cond = eng.unfold_features(eng.feature_encode(batch, st, 1, m0))
            x = batch["p1_face"][:, st, :].to(eng.theta.device).float().contiguous()
            eng.refresh(False)
            h = [None] * eng.K
            for k, layer in enumerate(self.glow.flow.layers):
                layer.actnorm.initialize_parameters(x)
                x, _, _, _, _ = eng.flowstep(k, x, cond, None, None, None, False, refresh=False)

    def forward(self, batch):
        eng = self.engine()
        self.glow.init_rnn_hidden()
        x0 = batch["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        Tp = T - eng.start_ts
        masks = self._masks(Tp, B, eng.theta.device)
        if self.training and not all(l.actnorm.inited for l in self.glow.flow.layers):
            self._ddi(eng, batch, masks)
        scale_out = None
        if self.hparams.Validation["scale_logging"] and eng.affine:
            scale_out = torch.empty(eng.K, B, eng.Cz, device=eng.theta.device)
        # Streams that require grad enter the autograd node as inputs (lfi_seq_train_bwd_dx gives their gradients).  They are
        # converted and cut to T frames here, with torch ops, so that the gradient flows back through the dtype / device copy
        # and the slice; the engine then finds them ready and reads them in place.
        mods, streams = (), ()
        if torch.is_grad_enabled():
            mods = tuple(i for i, m in enumerate(MODALITIES)
                         if eng.shape.hist[i] > 0 and isinstance(batch.get(m), torch.Tensor) and batch[m].requires_grad)
        if mods:
            batch = dict(batch)
            for i in mods:
                x = batch[MODALITIES[i]].to(device=eng.theta.device, dtype=torch.float32)
                if i > 0 and x.dim() == 3 and x.shape[1] > T:
                    x = x[:, :T]
                batch[MODALITIES[i]] = x.contiguous()
            streams = tuple(batch[MODALITIES[i]] for i in mods)
        z, nll = _SeqGlowFn.apply(eng, batch, masks, scale_out, mods, *streams, *eng.param_list())
        if scale_out is not None:
            for k, layer in enumerate(self.glow.flow.layers):
                layer.scale = scale_out[k]
        loss = nll.mean(dim=1).sum() / Tp
        losses = list(nll.detach().cpu().unbind(0))   # one device->host copy (the reference syncs every frame, models.py:554)
        z_seq = list(z.detach().unbind(0))
        return z_seq, loss.unsqueeze(-1), losses

    def evaluate(self, batch, chunk=None):
        """Likelihood of sequences of any length: returns what `with torch.no_grad(): forward(batch)` returns, (z_seq, loss [1],
        losses), with the same dropout masks (drawn in training mode, `injected_masks` when set), ActNorm initialisation and
        FlowStep.scale.  The frames are scored `chunk` at a time with the flow's RNN state carried from chunk to chunk, and nothing
        is kept for a backward pass, so memory does not grow with the sequence the way a no-grad `forward` does (that one lays out
        the training workspace).  chunk None: Engine.eval_chunk.  Always runs without autograd and returns detached tensors; use
        `forward` for gradients."""
        eng = self.engine()
        self.glow.init_rnn_hidden()
        with torch.no_grad():
            x0 = batch["p1_face"]
            B, T = x0.shape[0], x0.shape[1]
            Tp = T - eng.start_ts
            masks = self._masks(Tp, B, eng.theta.device)
            if self.training and not all(l.actnorm.inited for l in self.glow.flow.layers):
                self._ddi(eng, batch, masks)
            scale_out = None
            if self.hparams.Validation["scale_logging"] and eng.affine:
                scale_out = torch.empty(eng.K, B, eng.Cz, device=eng.theta.device)
            z, nll = eng.evaluate(batch, masks, chunk, scale_out)
            nll = nll - eng.logdet_const() / LN2
            if scale_out is not None:
                for k, layer in enumerate(self.glow.flow.layers):
                    layer.scale = scale_out[k]
            loss = nll.mean(dim=1).sum() / Tp
            losses = list(nll.cpu().unbind(0))  # one device->host copy
            return list(z.unbind(0)), loss.unsqueeze(-1), losses

    def loss(self, objective, z):
        """-(logdet + log N(z; 0, I)) / ln 2 per sample (models.py:563-565); mutates `objective` like the reference."""
        objective += GaussianDiag.logp_simplified(z)
        return (-objective) / float(np.log(2.0))

    def inference(self, seq_len, data=None, noise=None):
        """Autoregressive sampling (models.py:567-596): returns [B, seq_len - start_ts, C].
        `noise` [T',B,C] (already scaled by eps) replaces the drawn latent (parity tests)."""
        eng = self.engine()
        self.glow.init_rnn_hidden()
        with torch.no_grad():
            x0 = data["p1_face"]
            B = x0.shape[0]
            Tgen = seq_len - eng.start_ts
            eps = self.hparams.Infer["eps"]
            if noise is None and eps != 0:
                noise = torch.randn(Tgen, B, eng.C, device=eng.theta.device) * float(eps)
            faces, _ = eng.sample(data, seq_len, noise=noise, teacher_forced=False)
            return faces[:, eng.start_ts:]

    def create_conditioning(self, data, time_st, frame_nb, prev_p1_faces):
        """Feature vector of one frame (models.py:598-615)."""
        cond = self.hparams.Conditioning
        h0 = cond["p1_face"]["history"]
        output = {"prev_p1_face": prev_p1_faces[:, time_st - h0:time_st]}
        for modality in ["p1_speech", "p2_speech", "p2_face"]:
            history = cond[modality]["history"]
            if history:
                output[modality] = data[modality][:, (time_st - history) + 1:time_st + 1]
        self.engine()
        return self.feature_encoder(output)

    def invert(self, z_seq, data):
        """Inverse pass with given latents and teacher-forced conditioning (models.py:617-645)."""
        eng = self.engine()
        self.glow.init_rnn_hidden()
        with torch.no_grad():
            z = torch.stack([t.to(eng.theta.device).float() for t in z_seq])
            Tgen, B = z.shape[0], z.shape[1]
            seq_len = eng.start_ts + Tgen
            faces, ld = eng.sample(data, seq_len, noise=z, teacher_forced=True, want_logdet=True)
            logdet = ld - eng.logdet_const().detach()
            nll = GaussianDiag.nll_bits(z.reshape(Tgen * B, eng.C), logdet.reshape(Tgen * B)).view(Tgen, B)
            backward_loss = (nll.mean(dim=1).sum() / Tgen).unsqueeze(-1)
            rec = faces[:, eng.start_ts:].transpose(0, 1)
            return list(rec.unbind(0)), backward_loss
