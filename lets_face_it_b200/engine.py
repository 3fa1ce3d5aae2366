"""Engine: flat parameter storage + derived weight cache + workspaces behind the module API.

The reference modules own one small tensor per parameter and rebuild everything per frame
(SURVEY.md §2a).  Here all trainable tensors of the K flow steps and of the encoders live in ONE
flat fp32 buffer as `[K, ...]` blocks (what the kernels index), the `nn.Parameter`s of the module
tree are *views* into it (state-dict names/shapes unchanged, SURVEY.md §5), and gradients come
back as one flat buffer with the same layout (what NCCL all-reduces and the fused clip+Adam
consumes).  All compute goes through the C ABI (`_cabi.py`); there is no torch fallback.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, Optional

import torch

from . import _cabi as cabi

MODALITIES = ("p1_face", "p2_face", "p1_speech", "p2_speech")  # models.py:127-145 concat order
LN2 = math.log(2.0)

# (flat block name, attribute path below a FlowStep)
_STEP_BLOCKS_LU = [
    ("an_bias", "actnorm.bias"), ("an_logs", "actnorm.logs"),
    ("inv_l", "invconv.l"), ("inv_u", "invconv.u"), ("inv_log_s", "invconv.log_s"),
]
_STEP_BLOCKS_W = [("an_bias", "actnorm.bias"), ("an_logs", "actnorm.logs"), ("inv_w", "invconv.weight")]
_STEP_BLOCKS_F = [
    ("wc", "f.cond_transform.0.weight"), ("bc", "f.cond_transform.0.bias"),
    ("w_ih", "f.rnn.weight_ih"), ("b_ih", "f.rnn.bias_ih"), ("w_hh", "f.rnn.weight_hh"), ("b_hh", "f.rnn.bias_hh"),
    ("wf", "f.final_linear.weight"), ("bf", "f.final_linear.bias"), ("lf", "f.final_linear.logs"),
]
_ENC_BLOCKS = [("enc_w_ih", "weight_ih_l0"), ("enc_w_hh", "weight_hh_l0"), ("enc_b_ih", "bias_ih_l0"), ("enc_b_hh", "bias_hh_l0")]


def _get(mod, path):
    for p in path.split("."):
        mod = mod[int(p)] if p.isdigit() else getattr(mod, p)
    return mod


def _align(n, a=64):
    return (n + a - 1) // a * a


def _on_own_device(fn):
    """Runs an Engine method with the engine's device current: the C side launches on the current device and
    `cabi.stream_ptr()` is the current stream of the current device, while every pointer lives on `theta.device` (a model
    moved to cuda:1 without `torch.cuda.set_device(1)` would otherwise launch on device 0 against device 1 memory)."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **kw):
        self.ensure()  # (re)binds theta to the device the parameters live on now
        with torch.cuda.device(self.theta.device):
            return fn(self, *a, **kw)
    return wrapped


def feature_train_fwd(shape, P, bt, keep, t0, Tp, mode, dev):
    """lfi_feature_encode_fwd_train for a filled Params / Batch pair (`keep` holds the tensors they point into): returns
    (cond [Tp*B, Fe] folded, saved) with `saved` what `feature_train_bwd` needs (the stash included)."""
    L, st = cabi.lib(), cabi.stream_ptr()
    B, T = bt.B, bt.T
    cond = torch.empty(Tp * B, L.lfi_feature_dim_folded(ctypes.byref(shape)), dtype=torch.float32, device=dev)
    stash = torch.empty(max(256, L.lfi_feature_stash_bytes(ctypes.byref(shape), B, T, Tp, mode)), dtype=torch.uint8, device=dev)
    ws = torch.empty(max(256, L.lfi_feature_bwd_ws_bytes(ctypes.byref(shape), B, T, Tp, mode)), dtype=torch.uint8, device=dev)
    cabi.check(L.lfi_feature_encode_fwd_train(ctypes.byref(shape), ctypes.byref(P), ctypes.byref(bt), t0, Tp, cond.data_ptr(), stash.data_ptr(),
                                              stash.numel(), ws.data_ptr(), ws.numel(), mode, st), "lfi_feature_encode_fwd_train")
    return cond, (shape, P, bt, keep, t0, Tp, mode, stash)


def feature_train_bwd(saved, dcond, want_dx):
    """lfi_feature_encode_bwd: returns (dx, grads).  dx[i] = dL/d(stream i) [B, T, dim] or None where want_dx[i] is false or absent;
    grads[i] = (weight_ih, weight_hh, bias_ih, bias_hh) gradients of GRU modality i (written, not accumulated), None elsewhere."""
    shape, P, bt, keep, t0, Tp, mode, stash = saved
    L, st = cabi.lib(), cabi.stream_ptr()
    B, T = bt.B, bt.T
    dev = stash.device
    dcond = dcond.to(dtype=torch.float32).contiguous()
    dx, grads = [None] * cabi.NMOD, [None] * cabi.NMOD
    DX = (ctypes.c_void_p * cabi.NMOD)()
    G = cabi.Params()
    for i in range(cabi.NMOD):
        h, d, E = shape.hist[i], shape.dim[i], shape.ehid[i]
        if h > 0 and i < len(want_dx) and want_dx[i]:
            dx[i] = torch.empty(B, T, d, dtype=torch.float32, device=dev)
            DX[i] = dx[i].data_ptr()
        if h > 0 and E > 0:
            grads[i] = (torch.empty(3 * E, d, device=dev), torch.empty(3 * E, E, device=dev), torch.empty(3 * E, device=dev),
                        torch.empty(3 * E, device=dev))
            G.enc_w_ih[i], G.enc_w_hh[i], G.enc_b_ih[i], G.enc_b_hh[i] = [t.data_ptr() for t in grads[i]]
    ws = torch.empty(max(256, L.lfi_feature_bwd_ws_bytes(ctypes.byref(shape), B, T, Tp, mode)), dtype=torch.uint8, device=dev)
    cabi.check(L.lfi_feature_encode_bwd(ctypes.byref(shape), ctypes.byref(P), ctypes.byref(bt), t0, Tp, dcond.data_ptr(), DX, ctypes.byref(G),
                                        stash.data_ptr(), stash.numel(), ws.data_ptr(), ws.numel(), mode, st), "lfi_feature_encode_bwd")
    return dx, grads


class Engine:
    """One engine per top-level module (SeqGlow, or a stand-alone Glow/FlowNet/FlowStep)."""

    def __init__(self, steps, feature_encoder=None, gemm_mode=cabi.GEMM_FP32):
        self.steps = list(steps)
        self.fe = feature_encoder
        self.gemm_mode = gemm_mode
        self.theta: Optional[torch.Tensor] = None
        self.blocks: Dict[str, tuple] = {}      # name -> (offset, per-step numel or numel, K or 1)
        self._views: List[tuple] = []           # (param, offset, shape)
        self._ws: Dict[tuple, torch.Tensor] = {}
        self._derived = None
        self._fwd_token = 0
        self._derive_stream = None
        self._derive_event = None
        self.K = max(1, len(self.steps))
        if self.steps:
            s0 = self.steps[0]
            self.C = s0.actnorm.num_features
            self.H = s0.f.hidden_size
            self.D = s0.f.cond_transform[0].out_features
            self.F = s0.f.cond_transform[0].in_features
            self.G = 3 if s0.f.rnn_type == "gru" else 4
            self.LU = bool(s0.invconv.LU)
            self.affine = s0.flow_coupling == "affine"
            eps = float(s0.scale_eps)
        else:  # encoder-only engine (stand-alone FeatureEncoder): the flow fields are placeholders
            self.C, self.H, self.D, self.G, self.LU, self.affine, eps = feature_encoder._in_dim["p1_face"], 4, 4, 3, True, True, 1e-4
            self.F = feature_encoder.dim
        self.Ci, self.Cz = self.C // 2, self.C - self.C // 2
        self.Co = 2 * self.Cz if self.affine else self.Cz
        self.shape = cabi.Shape()
        sh = self.shape
        sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps = self.C, self.K, self.H, self.D, self.G, int(self.affine), eps
        if feature_encoder is None:
            sh.f_raw = self.F
            self.start_ts, self.Fe = 0, self.F
        else:
            sh.f_raw = 0
            for i, m in enumerate(MODALITIES):
                info = feature_encoder.modality_info(m)
                sh.hist[i], sh.dim[i], sh.ehid[i] = info
            L = cabi.lib()
            if L.lfi_feature_dim(ctypes.byref(sh)) < 0:
                raise RuntimeError("unsupported shape: %s" % L.lfi_last_error().decode())
            if L.lfi_feature_dim(ctypes.byref(sh)) != self.F:
                raise RuntimeError("feature encoder dim %d != cond_transform input %d (use_frame_nb / lstm / mlp / cnn encoders are "
                                   "outside the accelerated path, SURVEY.md §2 row 5)" % (L.lfi_feature_dim(ctypes.byref(sh)), self.F))
            self.start_ts = L.lfi_start_ts(ctypes.byref(sh))
            self.Fe = L.lfi_feature_dim_folded(ctypes.byref(sh))
        for k, st in enumerate(self.steps):
            st._engine, st._k = self, k

    # ------------------------------------------------------------------ flat storage
    def _layout(self):
        items = []  # (name, [params per step] or [param])
        # Order = the order in which the backward pass finishes the gradients: the flow-step weight blocks first (final before
        # the encoder backward: the bucket that is all-reduced while the encoders run), then ActNorm / 1x1-conv and the encoder
        # blocks (final only when the backward call returns) as ONE contiguous tail - a single trailing all-reduce.
        sb = _STEP_BLOCKS_F + (_STEP_BLOCKS_LU if self.LU else _STEP_BLOCKS_W)
        for name, path in sb:
            if self.steps:
                items.append((name, [_get(st, path) for st in self.steps]))
        if self.fe is not None:
            for i, m in enumerate(MODALITIES):
                enc = self.fe.gru_of(m)
                if enc is None:
                    continue
                for name, attr in _ENC_BLOCKS:
                    items.append(("%s.%d" % (name, i), [getattr(enc, attr)]))
        return items

    def ensure(self, device=None):
        """(Re)builds the flat buffer if the module parameters do not alias it (first use, .to(), ...)."""
        p0 = self.steps[0].actnorm.bias if self.steps else next(self.fe.parameters())
        device = device or p0.device
        if device.type != "cuda":
            raise RuntimeError("lets_face_it_b200: parameters live on %s; the flow runs on CUDA only (no CPU path)" % device)
        if self.theta is not None and self.theta.device == device:
            ok = all(p.data_ptr() == self.theta.data_ptr() + 4 * off and p.device == device for p, off, _ in self._views)
            if ok:
                return
        items = self._layout()
        off, blocks, views = 0, {}, []
        for name, plist in items:
            n = plist[0].numel()
            blocks[name] = (off, n, len(plist))
            for k, p in enumerate(plist):
                views.append((p, off + k * n, tuple(p.shape)))
            off = _align(off + n * len(plist))
        theta = torch.empty(off, dtype=torch.float32, device=device)
        theta.zero_()
        with torch.no_grad():
            for p, o, shp in views:
                theta[o:o + p.numel()].view(shp).copy_(p.data.to(device=device, dtype=torch.float32))
                p.data = theta[o:o + p.numel()].view(shp)
                p.grad = None
        self.theta, self.blocks, self._views = theta, blocks, views
        self.n_theta = off
        # constants of the LU parametrisation (buffers, modules.py:137-138) and composed weights
        K, C = self.K, self.C
        self._lu_key = None
        self._sync_lu_buffers(device)
        self.W = torch.empty(K, C, C, dtype=torch.float32, device=device)
        self.Winv = torch.empty(K, C, C, dtype=torch.float32, device=device)
        self._derived = torch.empty(cabi.lib().lfi_derived_bytes(ctypes.byref(self.shape)), dtype=torch.uint8, device=device)
        self._ws.clear()

    def _sync_lu_buffers(self, device=None):
        """Stacks the LU constants `invconv.p` / `invconv.sign_s` (buffers, modules.py:137-138) into [K,C,C] / [K,C].
        They are not part of theta: `load_state_dict` (or `.to()`) after the engine exists replaces them behind its back, so
        every refresh() compares their (storage, version) and re-stacks when any changed."""
        if not (self.LU and self.steps):
            return
        key = tuple((st.invconv.p.data_ptr(), st.invconv.p._version, st.invconv.sign_s.data_ptr(), st.invconv.sign_s._version)
                    for st in self.steps)
        if key == self._lu_key:
            return
        device = device or self.theta.device
        self.perm = torch.stack([st.invconv.p.detach().to(device=device, dtype=torch.float32) for st in self.steps]).contiguous()
        self.sign_s = torch.stack([st.invconv.sign_s.detach().to(device=device, dtype=torch.float32) for st in self.steps]).contiguous()
        self._lu_key = key

    def block(self, name, flat=None):
        off, n, k = self.blocks[name]
        return (self.theta if flat is None else flat)[off:off + n * k]

    def new_flat_grad(self):
        """Flat gradient buffer: theta layout followed by dW [K,C,C] (grad of the composed 1x1 weights)."""
        return torch.zeros(self.n_theta + _align(self.K * self.C * self.C), dtype=torch.float32, device=self.theta.device)

    def _params_struct(self, flat, w):
        P = cabi.Params()
        base = flat.data_ptr()

        def at(name):
            return base + 4 * self.blocks[name][0] if name in self.blocks else None

        for f in ("an_bias", "an_logs", "wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf"):
            setattr(P, f, at(f))
        P.w = w.data_ptr()
        for name, _ in _ENC_BLOCKS:
            arr = getattr(P, name)
            for i in range(cabi.NMOD):
                key = "%s.%d" % (name, i)
                arr[i] = at(key) if key in self.blocks else None
        return P

    def _workspace(self, key, nbytes):
        """ONE grow-only buffer per kind (key[0]: "train", "sample", "feat", ...): a validation shape, a partial last batch
        or a different chunk reuses it when it is large enough and replaces it when it is not (a workspace per (B, T) key
        would keep several multi-GB buffers alive for the life of the model)."""
        kind = key[0]
        t = self._ws.get(kind)
        if t is None or t.numel() < nbytes:
            self._ws.pop(kind, None)
            t = None  # release the old buffer before allocating the larger one
            t = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.theta.device)
            self._ws[kind] = t
        return t

    # ------------------------------------------------------------------ derived state
    @_on_own_device
    def refresh(self, need_inverse=False):
        """Composes W (and W^-1) from the LU parameters and rebuilds the derived weight cache.
        Call after every parameter change (done at the top of each forward / inference)."""
        self.ensure()
        self._sync_lu_buffers()
        L, st = cabi.lib(), cabi.stream_ptr()
        K, C = self.K, self.C
        if self.LU:
            ws = self._workspace(("invconv",), L.lfi_invconv_ws_bytes(K, C))
            cabi.check(L.lfi_invconv_compose(K, C, self.perm.data_ptr(), self.block("inv_l").data_ptr(), self.block("inv_u").data_ptr(),
                                             self.block("inv_log_s").data_ptr(), self.sign_s.data_ptr(), self.W.data_ptr(),
                                             self.Winv.data_ptr() if need_inverse else None, ws.data_ptr(), ws.numel(), st),
                       "lfi_invconv_compose")
        else:
            self.W.copy_(self.block("inv_w").view(K, C, C))
            if need_inverse:  # modules.py:155-160: inverse(weight.double()).float()
                self.Winv.copy_(torch.inverse(self.W.double()).float())
        P = self._params_struct(self.theta, self.W)
        cabi.check(L.lfi_derive(ctypes.byref(self.shape), ctypes.byref(P), self.Winv.data_ptr() if need_inverse else None,
                                self._derived.data_ptr(), self.gemm_mode, st), "lfi_derive")
        return P

    def logdet_const(self):
        """C * sum_k (sum logs_k + sum log|s_k|): the parameter-only part of every frame's log-det
        (modules.py:62 and :152/:171 — both multiply by input.size(1) = C)."""
        s = self.block("an_logs").sum()
        if self.LU:
            s = s + self.block("inv_log_s").sum()
        else:
            s = s + torch.slogdet(self.block("inv_w").view(self.K, self.C, self.C))[1].sum()
        return s * float(self.C)

    def step_logdet_const(self, k):
        st = self.steps[k]
        s = st.actnorm.logs.detach().sum()
        s = s + (st.invconv.log_s.detach().sum() if self.LU else torch.slogdet(st.invconv.weight.detach())[1])
        return s * float(self.C)

    # ------------------------------------------------------------------ batches
    def _batch_struct(self, data, B, T, masks=None, keep=None):
        bt = cabi.Batch()
        bt.B, bt.T = B, T
        keep = keep if keep is not None else []
        for i, m in enumerate(MODALITIES):
            x = data.get(m) if (self.shape.hist[i] > 0) else None
            if x is not None:
                x = x.to(device=self.theta.device, dtype=torch.float32).contiguous()
                if x.shape[0] != B or x.shape[2] != self.shape.dim[i]:
                    raise RuntimeError("batch[%s] has shape %s, expected [%d, T, %d]" % (m, tuple(x.shape), B, self.shape.dim[i]))
                if i > 0 and x.shape[1] != T:
                    x = x[:, :T].contiguous() if x.shape[1] > T else x
                    if x.shape[1] != T:
                        raise RuntimeError("batch[%s] has %d frames, expected %d" % (m, x.shape[1], T))
                keep.append(x)
                bt.x[i] = x.data_ptr()
            else:
                bt.x[i] = None
            mk = masks.get(m) if masks else None
            if mk is not None:
                mk = mk.to(device=self.theta.device, dtype=torch.float32).contiguous()
                keep.append(mk)
                bt.mask[i] = mk.data_ptr()
            else:
                bt.mask[i] = None
        return bt, keep

    # ------------------------------------------------------------------ SeqGlow.forward / backward
    @_on_own_device
    def train_forward(self, batch, masks=None, scale_out=None):
        """Returns (z [T',B,C], nll_core [T',B]); nll_core lacks the parameter-only log-det constant."""
        L = cabi.lib()
        dev = self.theta.device
        # The derived cache (composed 1x1 weights, folded W_c, transposes: ~25 short launches) is rebuilt on a side stream: the
        # conditioning encoders, which open the forward call, do not read it, and the call waits for the event only in front
        # of its first consumer (lfi_set_derived_ready_event).
        if self._derive_stream is None or self._derive_stream.device != dev:
            self._derive_stream = torch.cuda.Stream(device=dev)
            self._derive_event = torch.cuda.Event()
        side = self._derive_stream
        side.wait_stream(torch.cuda.current_stream(dev))  # after the optimizer update, and after every reader of the old cache
        with torch.cuda.stream(side):
            P = self.refresh(False)
            self._derive_event.record(side)
        ready = self._derive_event
        st = cabi.stream_ptr()
        x0 = batch["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        Tp = T - self.start_ts
        if Tp < 1:
            raise AssertionError("Sequence length %d must exceed the longest history %d (utils.py:116-122)" % (T, self.start_ts))
        bt, keep = self._batch_struct(batch, B, T, masks)
        dev = self.theta.device
        z = torch.empty(Tp, B, self.C, dtype=torch.float32, device=dev)
        nll = torch.empty(Tp, B, dtype=torch.float32, device=dev)
        ws = self._workspace(("train", B, T), L.lfi_train_ws_bytes(ctypes.byref(self.shape), B, T, self.gemm_mode))
        L.lfi_set_derived_ready_event(ready.cuda_event)
        try:
            rc = L.lfi_seq_train_fwd(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), ctypes.byref(bt),
                                     z.data_ptr(), nll.data_ptr(), scale_out.data_ptr() if scale_out is not None else None,
                                     ws.data_ptr(), ws.numel(), self.gemm_mode, st)
        finally:
            L.lfi_set_derived_ready_event(None)
            torch.cuda.current_stream(dev).wait_event(ready)  # (a failed call may not have consumed it)
        cabi.check(rc, "lfi_seq_train_fwd")
        self._fwd_token += 1
        self._last = (bt, keep, B, T, P)
        return z, nll

    @_on_own_device
    def train_backward(self, z, dnll, gflat, token=None, dx=None):
        """Accumulates dL/dtheta into gflat (layout of new_flat_grad) given dL/dnll [T',B].  dx: None, or one entry per modality,
        None or a [B, T, dim] fp32 tensor that receives dL/d(stream) (lfi_seq_train_bwd_dx; written, not accumulated)."""
        if token is not None and token != self._fwd_token:
            raise RuntimeError("backward called after another forward on the same engine: the activation stash was overwritten")
        L, st = cabi.lib(), cabi.stream_ptr()
        bt, keep, B, T, P = self._last
        dW = gflat[self.n_theta:self.n_theta + self.K * self.C * self.C]
        Gs = self._params_struct(gflat, dW)
        dnll = dnll.to(dtype=torch.float32).contiguous()
        ws = self._workspace(("train", B, T), 0)
        if dx is None:
            cabi.check(L.lfi_seq_train_bwd(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), ctypes.byref(bt),
                                           z.data_ptr(), dnll.data_ptr(), ctypes.byref(Gs), ws.data_ptr(), ws.numel(), self.gemm_mode, st),
                       "lfi_seq_train_bwd")
        else:
            DX = (ctypes.c_void_p * cabi.NMOD)(*[cabi.ptr(t) for t in dx])
            dws = self._workspace(("train_dx",), L.lfi_train_dx_ws_bytes(ctypes.byref(self.shape), B, T, self.gemm_mode))
            cabi.check(L.lfi_seq_train_bwd_dx(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), ctypes.byref(bt),
                                              z.data_ptr(), dnll.data_ptr(), ctypes.byref(Gs), ws.data_ptr(), ws.numel(), DX,
                                              dws.data_ptr(), dws.numel(), self.gemm_mode, st), "lfi_seq_train_bwd_dx")
        # the parameter-only constant: nll -= C * (sum logs + sum log_s) / ln2   for every (t, b)
        coef = -(float(self.C) / LN2) * dnll.sum()
        self.block("an_logs", gflat).add_(coef)
        if self.LU:
            self.block("inv_log_s", gflat).add_(coef)
            wsi = self._workspace(("invconv",), L.lfi_invconv_ws_bytes(self.K, self.C))
            cabi.check(L.lfi_invconv_compose_bwd(self.K, self.C, self.perm.data_ptr(), self.block("inv_l").data_ptr(),
                                                 self.block("inv_u").data_ptr(), self.block("inv_log_s").data_ptr(),
                                                 self.sign_s.data_ptr(), dW.data_ptr(), self.block("inv_l", gflat).data_ptr(),
                                                 self.block("inv_u", gflat).data_ptr(), self.block("inv_log_s", gflat).data_ptr(),
                                                 wsi.data_ptr(), wsi.numel(), st), "lfi_invconv_compose_bwd")
        else:
            W = self.block("inv_w").view(self.K, self.C, self.C)
            g = self.block("inv_w", gflat).view(self.K, self.C, self.C)
            g.add_(dW.view(self.K, self.C, self.C))
            g.add_(coef * torch.inverse(W.double()).float().transpose(1, 2))  # d log|det W| / dW = W^-T
        return gflat

    def grad_views(self, gflat):
        """Per-parameter views of a flat gradient, in the order of `self.param_list()`."""
        return [gflat[o:o + p.numel()].view(shp) for p, o, shp in self._views]

    def param_list(self):
        self.ensure()
        return [p for p, _, _ in self._views]

    # ------------------------------------------------------------------ SeqGlow.evaluate
    def eval_chunk(self, B, T):
        """Default frames per chunk of `evaluate`: as many as keep the chunk-dependent part of its workspace within 2.5 GB, so that
        a training window (56 frames at B = 256, 2.2 GB in bf16x3 at final_model.yaml shapes) is one chunk.  Shorter chunks spend
        a growing share of the time in the flow-core pipeline's fill and drain (K - 1 stage periods per chunk)."""
        Tp = T - self.start_ts
        if Tp <= 8:
            return max(1, Tp)
        L = cabi.lib()
        size = lambda c: L.lfi_eval_ws_bytes(ctypes.byref(self.shape), B, T, c, self.gemm_mode)
        per_frame = max(1.0, (size(8) - size(1)) / 7.0)
        return max(1, min(Tp, int(2.5e9 // per_frame)))

    @_on_own_device
    def evaluate(self, batch, masks=None, chunk=None, scale_out=None):
        """Returns (z [T',B,C], nll_core [T',B]) as train_forward does, without gradients: the frames are scored `chunk` at a time
        (lfi_seq_eval) and nothing is kept for a backward pass, so the workspace does not grow with T except for the encoders'
        per-raw-frame input projections.  nll_core lacks the parameter-only log-det constant."""
        P = self.refresh(False)
        L, st = cabi.lib(), cabi.stream_ptr()
        dev = self.theta.device
        x0 = batch["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        Tp = T - self.start_ts
        if Tp < 1:
            raise AssertionError("Sequence length %d must exceed the longest history %d (utils.py:116-122)" % (T, self.start_ts))
        chunk = self.eval_chunk(B, T) if chunk is None else int(chunk)
        if chunk < 1:
            raise ValueError("chunk must be >= 1, got %d" % chunk)
        bt, keep = self._batch_struct(batch, B, T, masks)
        z = torch.empty(Tp, B, self.C, dtype=torch.float32, device=dev)
        nll = torch.empty(Tp, B, dtype=torch.float32, device=dev)
        ws = self._workspace(("eval",), L.lfi_eval_ws_bytes(ctypes.byref(self.shape), B, T, chunk, self.gemm_mode))
        cabi.check(L.lfi_seq_eval(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), ctypes.byref(bt), chunk,
                                  z.data_ptr(), nll.data_ptr(), scale_out.data_ptr() if scale_out is not None else None,
                                  ws.data_ptr(), ws.numel(), self.gemm_mode, st), "lfi_seq_eval")
        return z, nll

    # ------------------------------------------------------------------ SeqGlow.inference / invert
    @_on_own_device
    def sample(self, data, seq_len, noise=None, teacher_forced=False, chunk=None, want_logdet=False):
        """faces [B, seq_len, C]: seed in [:, :start_ts], generated (or reconstructed) frames after."""
        P = self.refresh(True)
        L, st = cabi.lib(), cabi.stream_ptr()
        dev = self.theta.device
        x0 = data["p1_face"].to(device=dev, dtype=torch.float32)
        B = x0.shape[0]
        Tgen = seq_len - self.start_ts
        if Tgen < 1:
            raise AssertionError("seq_len %d must exceed the longest history %d" % (seq_len, self.start_ts))
        T = None
        for i, m in enumerate(MODALITIES[1:], 1):
            if self.shape.hist[i] > 0:
                if data[m].shape[1] < seq_len:
                    raise RuntimeError("data[%s] has %d frames, need seq_len=%d" % (m, data[m].shape[1], seq_len))
                T = seq_len
        T = T or seq_len
        d2 = dict(data)
        for m in MODALITIES[1:]:
            if m in d2 and d2[m] is not None:
                d2[m] = d2[m][:, :seq_len]
        faces = torch.zeros(B, seq_len, self.C, dtype=torch.float32, device=dev)
        if teacher_forced:
            if x0.shape[1] < seq_len:
                raise RuntimeError("invert needs data['p1_face'] with >= %d frames" % seq_len)
            d2["p1_face"] = x0[:, :seq_len]
        else:
            if x0.shape[1] < self.start_ts:
                raise RuntimeError("inference needs %d seed frames in data['p1_face']" % self.start_ts)
            faces[:, :self.start_ts] = x0[:, :self.start_ts]
            d2["p1_face"] = None
        bt, keep = self._batch_struct({k: v for k, v in d2.items() if v is not None}, B, T)
        if chunk is None:
            # bound the chunk's static cond_transform block (Mc x K*D fp32) to ~1.5 GB
            chunk = max(1, min(Tgen, int(1.5e9 // max(1, B * self.K * self.D * 4))))
        if noise is not None:
            noise = noise.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(noise.shape) != (Tgen, B, self.C):
                raise RuntimeError("noise must be [%d, %d, %d], got %s" % (Tgen, B, self.C, tuple(noise.shape)))
        logdet = torch.zeros(Tgen, B, dtype=torch.float32, device=dev) if want_logdet else None
        ws = self._workspace(("sample", B, T, chunk), L.lfi_sample_ws_bytes(ctypes.byref(self.shape), B, T, chunk, self.gemm_mode))
        cabi.check(L.lfi_seq_sample(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), ctypes.byref(bt), seq_len,
                                    noise.data_ptr() if noise is not None else None, faces.data_ptr(),
                                    logdet.data_ptr() if logdet is not None else None, int(teacher_forced), int(chunk),
                                    ws.data_ptr(), ws.numel(), self.gemm_mode, st), "lfi_seq_sample")
        return faces, logdet

    # ------------------------------------------------------------------ module-level API
    @_on_own_device
    def feature_encode(self, data, t0, Tp, masks=None):
        """Folded FeatureEncoder output [Tp*B, Fe] for frames t0..t0+Tp-1 of a batch dict."""
        self.ensure()
        L, st = cabi.lib(), cabi.stream_ptr()
        P = self._params_struct(self.theta, self.W)
        x0 = data["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        bt, keep = self._batch_struct(data, B, T, masks)
        cond = torch.empty(Tp * B, self.Fe, dtype=torch.float32, device=self.theta.device)
        ws = self._workspace(("feat", B, T, Tp), L.lfi_feature_ws_bytes(ctypes.byref(self.shape), B, T, Tp, self.gemm_mode))
        cabi.check(L.lfi_feature_encode(ctypes.byref(self.shape), ctypes.byref(P), ctypes.byref(bt), t0, Tp, cond.data_ptr(),
                                        ws.data_ptr(), ws.numel(), self.gemm_mode, st), "lfi_feature_encode")
        return cond

    @_on_own_device
    def feature_encode_train(self, data, t0, Tp, masks=None):
        """`feature_encode` with the stash `feature_encode_backward` needs (lfi_feature_encode_fwd_train): (cond, saved)."""
        self.ensure()
        P = self._params_struct(self.theta, self.W)
        x0 = data["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        bt, keep = self._batch_struct(data, B, T, masks)
        return feature_train_fwd(self.shape, P, bt, keep, t0, Tp, self.gemm_mode, self.theta.device)

    @_on_own_device
    def feature_encode_backward(self, saved, dcond, want_dx):
        """Backward of `feature_encode_train` (lfi_feature_encode_bwd): dL/d(stream) [B, T, dim] per modality (None where
        want_dx[i] is false) and the encoder gradients as `feature_train_bwd` returns them."""
        return feature_train_bwd(saved, dcond, want_dx)

    def unfold_features(self, cond):
        """[M, Fe] folded -> [M, F] as the reference lays it out (GRU state concatenated twice, models.py:64)."""
        parts, off = [], 0
        for i, m in enumerate(MODALITIES):
            h, dmm, e = self.shape.hist[i], self.shape.dim[i], self.shape.ehid[i]
            if h <= 0:
                continue
            w = e if e > 0 else h * dmm
            blk = cond[:, off:off + w]
            parts.extend([blk, blk] if e > 0 else [blk])
            off += w
        return torch.cat(parts, dim=1)

    @_on_own_device
    def flowstep(self, k, x, cond, h_in, c_in, logdet, reverse, want_scale=False, refresh=True):
        """One FlowStep on one frame (models.py:305-373).  Returns (y, logdet, h, c, scale)."""
        if refresh:
            self.refresh(reverse)
        L, st = cabi.lib(), cabi.stream_ptr()
        P = self._params_struct(self.theta, self.W)
        dev = self.theta.device
        x = x.to(device=dev, dtype=torch.float32).contiguous()
        cond = cond.to(device=dev, dtype=torch.float32).contiguous()
        B = x.shape[0]
        if x.shape[1] != self.C or cond.shape[1] != self.F:
            raise RuntimeError("flow step expects x [B,%d] and cond [B,%d], got %s / %s" % (self.C, self.F, tuple(x.shape), tuple(cond.shape)))
        y = torch.empty_like(x)
        h_out = torch.empty(B, self.H, dtype=torch.float32, device=dev)
        c_out = torch.empty(B, self.H, dtype=torch.float32, device=dev) if self.G == 4 else None
        ld = torch.zeros(B, dtype=torch.float32, device=dev)
        scale = torch.empty(B, self.Cz, dtype=torch.float32, device=dev) if (want_scale and not reverse and self.affine) else None
        ws = self._workspace(("step", B), L.lfi_flowstep_ws_bytes(ctypes.byref(self.shape), B))
        cabi.check(L.lfi_flowstep(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), k, int(reverse), x.data_ptr(),
                                  cond.data_ptr(), cabi.ptr(h_in), cabi.ptr(c_in), h_out.data_ptr(),
                                  c_out.data_ptr() if c_out is not None else None, y.data_ptr(), ld.data_ptr(),
                                  scale.data_ptr() if scale is not None else None, B, ws.data_ptr(), ws.numel(), st), "lfi_flowstep")
        if logdet is not None:
            const = self.step_logdet_const(k)
            logdet = logdet + (ld - const if reverse else ld + const)
        return y, logdet, h_out, c_out, scale

    # ------------------------------------------------------------------ FlowStep.forward under autograd
    _STEP_GRAD_BLOCKS = ("an_bias", "an_logs", "w", "wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf")

    def _step_block_numel(self):
        C, D, F, GH, H, Co, In = self.C, self.D, self.F, self.G * self.H, self.H, self.Co, self.Ci + self.D
        return {"an_bias": C, "an_logs": C, "w": C * C, "wc": D * F, "bc": D, "w_ih": GH * In, "b_ih": GH, "w_hh": GH * H, "b_hh": GH,
                "wf": Co * H, "bf": Co, "lf": Co}

    @_on_own_device
    def flowstep_train(self, k, x, cond, h_in, c_in, want_scale=False, refresh=True, reverse=False):
        """Forward of one FlowStep on one frame WITH the stash `flowstep_backward` needs (lfi_flowstep_fwd_train; reverse=True:
        lfi_flowstep_rev_fwd_train, which has no scale).  Returns (y, ld [B] coupling log-det term, h_out, c_out, scale, stash).
        refresh=False: the derived cache is current (FlowNet.encode / decode rebuild it once per call)."""
        if refresh:
            self.refresh(reverse)
        L, st = cabi.lib(), cabi.stream_ptr()
        P = self._params_struct(self.theta, self.W)
        dev = self.theta.device
        x = x.detach().to(device=dev, dtype=torch.float32).contiguous()
        cond = cond.detach().to(device=dev, dtype=torch.float32).contiguous()
        h_in = h_in.detach().to(device=dev, dtype=torch.float32).contiguous() if h_in is not None else None
        c_in = c_in.detach().to(device=dev, dtype=torch.float32).contiguous() if c_in is not None else None
        B = x.shape[0]
        if x.shape[1] != self.C or cond.shape[1] != self.F:
            raise RuntimeError("flow step expects x [B,%d] and cond [B,%d], got %s / %s" % (self.C, self.F, tuple(x.shape), tuple(cond.shape)))
        y = torch.empty_like(x)
        h_out = torch.empty(B, self.H, dtype=torch.float32, device=dev)
        c_out = torch.empty(B, self.H, dtype=torch.float32, device=dev) if self.G == 4 else None
        ld = torch.zeros(B, dtype=torch.float32, device=dev)
        scale = torch.empty(B, self.Cz, dtype=torch.float32, device=dev) if (want_scale and self.affine and not reverse) else None
        stash = torch.empty(L.lfi_flowstep_stash_bytes(ctypes.byref(self.shape), B), dtype=torch.uint8, device=dev)
        ws = self._workspace(("step", B), L.lfi_flowstep_ws_bytes(ctypes.byref(self.shape), B))
        if reverse:
            cabi.check(L.lfi_flowstep_rev_fwd_train(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), k, x.data_ptr(),
                                                    cond.data_ptr(), cabi.ptr(h_in), cabi.ptr(c_in), h_out.data_ptr(), cabi.ptr(c_out),
                                                    y.data_ptr(), ld.data_ptr(), B, stash.data_ptr(), stash.numel(), ws.data_ptr(), ws.numel(),
                                                    st), "lfi_flowstep_rev_fwd_train")
            return y, ld, h_out, c_out, scale, (stash, cond, h_in, c_in)
        cabi.check(L.lfi_flowstep_fwd_train(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), k, x.data_ptr(), cond.data_ptr(),
                                            cabi.ptr(h_in), cabi.ptr(c_in), h_out.data_ptr(), c_out.data_ptr() if c_out is not None else None,
                                            y.data_ptr(), ld.data_ptr(), scale.data_ptr() if scale is not None else None, B,
                                            stash.data_ptr(), stash.numel(), ws.data_ptr(), ws.numel(), st), "lfi_flowstep_fwd_train")
        return y, ld, h_out, c_out, scale, (stash, cond, h_in, c_in)

    @_on_own_device
    def flowstep_backward(self, k, saved, dy, dld, dh_out, dc_out, reverse=False):
        """Backward of `flowstep_train` (lfi_flowstep_bwd; reverse=True: lfi_flowstep_rev_bwd).  Returns (dx, dcond, dh_in, dc_in,
        grads) with grads a dict block name -> gradient tensor of step k's block (dW of the composed 1x1 weight under "w", in both
        directions)."""
        L, st = cabi.lib(), cabi.stream_ptr()
        stash, cond, h_in, c_in = saved
        dev = self.theta.device
        P = self._params_struct(self.theta, self.W)
        B = cond.shape[0]
        f32 = lambda t: t.detach().to(device=dev, dtype=torch.float32).contiguous() if t is not None else None
        dy = f32(dy) if dy is not None else torch.zeros(B, self.C, device=dev)
        dld, dh_out, dc_out = f32(dld), f32(dh_out), f32(dc_out)
        dx = torch.empty(B, self.C, dtype=torch.float32, device=dev)
        dcond = torch.empty(B, self.F, dtype=torch.float32, device=dev)
        dh_in = torch.empty(B, self.H, dtype=torch.float32, device=dev)
        dc_in = torch.empty(B, self.H, dtype=torch.float32, device=dev) if self.G == 4 else None
        numel = self._step_block_numel()
        offs, o = {}, 0
        for n in self._STEP_GRAD_BLOCKS:
            offs[n] = o
            o = _align(o + numel[n])
        gbuf = torch.zeros(o, dtype=torch.float32, device=dev)
        G = cabi.Params()
        for n in self._STEP_GRAD_BLOCKS:  # the C side indexes [K, ...] blocks: base moved back by k blocks
            setattr(G, n, gbuf.data_ptr() + 4 * offs[n] - 4 * k * numel[n])
        name, size = ("lfi_flowstep_rev_bwd", L.lfi_flowstep_rev_bwd_ws_bytes) if reverse else ("lfi_flowstep_bwd", L.lfi_flowstep_bwd_ws_bytes)
        ws = self._workspace(("stepbwd", B), size(ctypes.byref(self.shape), B))
        cabi.check(getattr(L, name)(ctypes.byref(self.shape), self._derived.data_ptr(), ctypes.byref(P), k, cond.data_ptr(), cabi.ptr(h_in),
                                    cabi.ptr(c_in), dy.data_ptr(), cabi.ptr(dld), cabi.ptr(dh_out), cabi.ptr(dc_out), dx.data_ptr(),
                                    dcond.data_ptr(), dh_in.data_ptr(), dc_in.data_ptr() if dc_in is not None else None, ctypes.byref(G), B,
                                    stash.data_ptr(), stash.numel(), ws.data_ptr(), ws.numel(), st), name)
        grads = {n: gbuf[offs[n]:offs[n] + numel[n]] for n in self._STEP_GRAD_BLOCKS}
        return dx, dcond, dh_in, dc_in, grads

    @_on_own_device
    def invconv_chain_rule(self, k, dW):
        """dL/d(l, u, log_s) of step k from dL/dW of its composed weight (lfi_invconv_compose_bwd on one step)."""
        L, st = cabi.lib(), cabi.stream_ptr()
        C, dev = self.C, self.theta.device
        n = C * C
        blk = lambda name, m: self.block(name)[k * m:(k + 1) * m]
        dl = torch.zeros(C, C, device=dev)
        du = torch.zeros(C, C, device=dev)
        dls = torch.zeros(C, device=dev)
        ws = self._workspace(("invconv1",), L.lfi_invconv_ws_bytes(1, C))
        cabi.check(L.lfi_invconv_compose_bwd(1, C, self.perm[k].contiguous().data_ptr(), blk("inv_l", n).data_ptr(), blk("inv_u", n).data_ptr(),
                                             blk("inv_log_s", C).data_ptr(), self.sign_s[k].contiguous().data_ptr(), dW.contiguous().data_ptr(),
                                             dl.data_ptr(), du.data_ptr(), dls.data_ptr(), ws.data_ptr(), ws.numel(), st),
                   "lfi_invconv_compose_bwd")
        return dl, du, dls
