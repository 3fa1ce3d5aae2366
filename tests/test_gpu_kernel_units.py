"""Direct unit tests of the tcgen05 GEMM's internal epilogues and the encoder-GRU kernels against fp64 references.

The production C ABI reaches gemm_tc only with fp32 operands and the generic epilogues (tests/test_gpu_gemm_tc.py).  The
training step and the sampler also use operand planes, plane outputs, the sign-of-plane LeakyReLU', fused column sums,
the row-interleaved output, the scalar epilogue with split-K atomics, the fused encoder-GRU epilogues and the encoder aux
kernels.  These tests drive them through the test-only probe library (tests/kernel_probe.py), which calls the internal
functions of the shipped liblfi_b200.so with the argument combinations seq.cu issues, at the final_model.yaml shapes:
C 56, K 16, H 128, GH 384, D 512, Fe 920, Far 280, encoders E/hist/dim 256/24/56, 128/2/30, 256/16/30.  Rows are
M = B * T' with T' = 56 (T = 80 minus the 24 history frames): B = 256 -> 14,336 rows (a multiple of 128), B = 100 ->
5,600 rows (a ragged last 128-row tile).

Every reference is computed in fp64 on the GPU from the same fp32 operands the planes were split from.  Tolerances:
  * GEMM outputs: 3e-5 (bf16x3) and 1.5e-2 (bf16) of max|ref|, the bounds tests/test_gpu_gemm_tc.py states for the same
    kernel.  They are applied per batch slice and per 128-row tile (max error in the tile over max|ref| in the tile), so an
    error confined to one tile or slice cannot hide under the others.  Sharpness: every bf16x3 case also runs in bf16 and
    asserts that this error EXCEEDS 3e-5, i.e. the check would notice a dropped hi*lo correction product.
  * Long reductions (weight gradients over K rows): the fp32 accumulation adds a random walk of sqrt(K) * 2^-24 of the
    result on top of the operand error; the 3e-5 bound was stated for K <= 14,080, so these cases use
    3e-5 + sqrt(K) * 2^-24 (3.7e-5 at K = 14,336, 5.8e-5 at K = 215,040).
  * GRU h / gates / cond: 1e-4 of max|ref| in bf16x3, as the encoder checks of tests/test_gpu_paths.py.  In bf16 mode the
    pre-activations carry the bf16 GEMM bound (1.5e-2 of their max); sigmoid and tanh are at most 1-Lipschitz and
    h = n + u (h_prev - n) adds at most a quarter of the u error, so h and the gates are bounded by 1.25 * 1.5e-2 of the
    pre-activations' max|a| per tile.
  * Aux kernels whose inputs are exact fp32 (no bf16 operand): 1e-5 of max|ref|.  They run about ten fp32 operations
    (expf / tanhf within 2 ulp) per output, i.e. errors near 1e-6; 1e-5 leaves a factor of ten.
  * Column sums accumulated with fp32 atomics: 1e-5 of sum|terms| per column.  A sum runs through at most ~1,000
    sequential fp32 additions (per-thread rows, the in-block reduction, one atomic per block); with random-signed rounding
    that is sqrt(1000) * 2^-24 = 2e-6 of sum|terms|.  One missing row of 5,600 moves a sum by ~2e-4 of sum|terms|.
  * Exact properties (plane splits, layout permutations, the same value written twice): bitwise.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests import kernel_probe as kp

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF16X3, BF16 = 1, 2
MODES = [("bf16x3", BF16X3, 3e-5), ("bf16", BF16, 1.5e-2)]
GRU_TOL = {BF16X3: 1e-4, BF16: 5e-3}      # of max|ref| (the persistent encoder: h after all window steps)
STEP_TOL = {BF16X3: 1e-4, BF16: 1.25 * 1.5e-2}  # one fused step; bf16: of the pre-activations' max (module docstring)
EXACT_TOL = 1e-5
SUM_TOL = 1e-5
EPI_BIAS, EPI_LRELU, EPI_ACCUM, EPI_LRELU_BWD = 1, 2, 4, 8

K_, H_, D_, CI, FE, FAR = 16, 128, 512, 28, 920, 280
GH = 3 * H_
IN = CI + D_
T_, T0, TP = 80, 24, 56
BATCHES = [256, 100]             # M = 14,336 (whole tiles) and 5,600 (ragged last tile)
ENCODERS = [(256, 24, 56), (128, 2, 30), (256, 16, 30)]  # E, hist, dim: p2_face, p1_speech, p2_speech


# ---- helpers -------------------------------------------------------------------------------------------------------
def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def randn(*shape, g, scale=1.0):
    return torch.randn(*shape, generator=g, device=DEV) * scale


def planes(x, ldp=None):
    """fp32 [..., cols] -> (hi, lo) bf16 [..., ldp] split as the library does: hi = bf16_rn(x), lo = bf16_rn(x - hi)."""
    if ldp is not None and ldp > x.shape[-1]:
        x = F.pad(x, (0, ldp - x.shape[-1]))
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return hi.contiguous(), lo.contiguous()


def pv(hi, lo):
    return hi.double() + lo.double()


def bits(t):
    return t.contiguous().view(torch.int16) if t.dtype == torch.bfloat16 else t.contiguous().view(torch.int32)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def lrelu(x):
    return torch.where(x > 0, x, 0.01 * x)


def tile_err(got, ref, scale=None):
    """max over batch slices and 128-row tiles of (max |got - ref| in the tile) / (max |scale| in the tile), scale = ref
    unless given."""
    if got.dim() == 2:
        got, ref = got[None], ref[None]
        scale = None if scale is None else scale[None]
    d = (got.double() - ref).abs()
    r = (ref if scale is None else scale).abs()
    pad = (-d.shape[1]) % 128
    d = F.pad(d, (0, 0, 0, pad)).reshape(d.shape[0], -1, 128 * d.shape[2]).amax(2)
    r = F.pad(r, (0, 0, 0, pad)).reshape(r.shape[0], -1, 128 * r.shape[2]).amax(2)
    return float((d / r.clamp_min(1e-30)).max())


def rel_err(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def sum_err(got, ref, absum):
    return float(((got.double() - ref).abs() / absum.clamp_min(1e-30)).max())


def P(t):
    return None if t is None else t.data_ptr()


def plane(hi, lo, ld, stride=0, off=0):
    return kp.PlaneRef(P(hi) + 2 * off, (P(lo) + 2 * off) if lo is not None else None, ld, stride)


def stream():
    return torch.cuda.current_stream().cuda_stream


def gemm(mode, tA, tB, M, N, K, **kw):
    L = kp.lib()
    g = kp.GemmArgs()
    g.transA, g.transB, g.M, g.N, g.K, g.batch = tA, tB, M, N, K, 1
    for k, v in kw.items():
        setattr(g, k, v)
    n = int(L.lfi_probe_gemm_ws_bytes(mode, C.byref(g)))
    ws = torch.empty(max(n, 1), dtype=torch.uint8, device=DEV)
    kp.check(L.lfi_probe_gemm(mode, C.byref(g), ws.data_ptr(), n, stream()), "gemm")
    torch.cuda.synchronize()


def check_modes(errs, what, K=None):
    """errs: {mode: error}.  Each mode within its bound, and the bf16 run beyond the bf16x3 bound (sharpness).  K: length
    of a long reduction (adds the fp32 accumulation term of the module docstring)."""
    tol = 3e-5 + (K ** 0.5 * 2.0 ** -24 if K else 0.0)
    assert errs[BF16X3] < tol, (what, "bf16x3", tol, errs)
    assert errs[BF16] < 1.5e-2, (what, "bf16", errs)
    assert errs[BF16] > 3e-5, (what, "bf16 run within the bf16x3 bound: the check could not see a dropped correction", errs)
    print(what, {("bf16x3" if m == BF16X3 else "bf16"): "%.2e" % e for m, e in errs.items()})


# ---- cond_transform: BIAS | LRELU, planes out only ---------------------------------------------------------------------
@pytest.mark.parametrize("B", BATCHES)
def test_cond_transform_plane_output(B):
    M, N, Kd = B * TP, K_ * D_, FE
    g = gen(1)
    A = randn(M, Kd, g=g)
    W = randn(N, Kd, g=g, scale=Kd ** -0.5)
    b = randn(N, g=g, scale=0.3)
    ref = lrelu(A.double() @ W.double().T + b.double())
    errs = {}
    for _, mode, _ in MODES:
        hi = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
        lo = torch.empty_like(hi)
        gemm(mode, 0, 1, M, N, Kd, A=P(A), lda=Kd, B=P(W), ldb=Kd, C=None, ldc=N, epi=EPI_BIAS | EPI_LRELU, bias=P(b),
             pOut=plane(hi, lo, N))
        errs[mode] = tile_err(pv(hi, lo), ref)
        # the planes are exactly the split of the fp32 value the same GEMM stores into C: hi = bf16_rn(C), lo = bf16_rn(C - hi).
        # (hi == bf16_rn(hi + lo) is not an invariant of this split: when C - hi lies just under half a bf16 ulp, lo rounds to
        # exactly half an ulp and hi + lo is a tie, which round-to-even may resolve away from hi.)
        Cf = torch.empty(M, N, device=DEV)
        gemm(mode, 0, 1, M, N, Kd, A=P(A), lda=Kd, B=P(W), ldb=Kd, C=P(Cf), ldc=N, epi=EPI_BIAS | EPI_LRELU, bias=P(b))
        assert same_bits(hi, Cf.to(torch.bfloat16))
        assert same_bits(lo, (Cf - hi.float()).to(torch.bfloat16))
        del hi, lo, Cf
    check_modes(errs, "cond_transform M=%d" % M)


# ---- gate-ih: plane column slices, batch K, BIAS, row-interleaved output ----------------------------------------------
@pytest.mark.parametrize("M", [256 * TP, 100 * TP, 100 * TP - 13])
def test_gate_ih_plane_slices_and_tiled_output(M):
    g = gen(2)
    cact = lrelu(randn(M, K_ * D_, g=g))
    chi, clo = planes(cact)
    w_ih = randn(K_, GH, IN, g=g, scale=IN ** -0.5)
    b_ih = randn(K_, GH, g=g, scale=0.3)
    ref = torch.stack([cact[:, k * D_:(k + 1) * D_].double() @ w_ih[k, :, CI:].double().T + b_ih[k].double() for k in range(K_)])
    Mp = (M + 31) // 32 * 32
    errs = {}
    for _, mode, _ in MODES:
        kw = dict(A=None, lda=K_ * D_, B=P(w_ih) + 4 * CI, ldb=IN, sB=GH * IN, epi=EPI_BIAS, bias=P(b_ih), sBias=GH,
                  batch=K_, pA=plane(chi, clo, K_ * D_, D_))
        Crm = torch.empty(M, K_ * GH, device=DEV)
        gemm(mode, 0, 1, M, GH, D_, C=P(Crm), ldc=K_ * GH, sC=GH, **kw)
        errs[mode] = tile_err(Crm.view(M, K_, GH).permute(1, 0, 2), ref)
        Ct = torch.full((Mp * K_ * GH,), float("nan"), device=DEV)
        gemm(mode, 0, 1, M, GH, D_, C=P(Ct), ldc=K_ * GH, sC=GH * 32, c_tiled32=1, **kw)
        # element (m, n) at ((m / 32) * (ldc / 4) + n / 4) * 128 + (m % 32) * 4 + n % 4: bitwise the row-major result
        untiled = Ct.view(Mp // 32, K_ * GH // 4, 32, 4).permute(0, 2, 1, 3).reshape(Mp, K_ * GH)
        assert same_bits(untiled[:M], Crm), "row-interleaved output differs from the row-major output of the same call"
        assert torch.isnan(untiled[M:]).all(), "rows beyond M written"
    check_modes(errs, "gate-ih M=%d" % M)


# ---- cond backward: planes in, planes out, LeakyReLU' from the sign of a bf16 plane, fused column sums -----------------
@pytest.mark.parametrize("B", BATCHES)
def test_cond_backward_auxp_colsum(B):
    M = B * TP
    g = gen(3)
    dG = randn(M, K_ * GH, g=g)
    ghi, glo = planes(dG)
    w_ih = randn(K_, GH, IN, g=g, scale=GH ** -0.5)
    cact = randn(M, K_ * D_, g=g)
    ahi, _ = planes(cact)
    bc0 = randn(K_, D_, g=g)
    slope = torch.where(ahi.float() > 0, 1.0, 0.01).double()
    prod = torch.stack([(dG[:, k * GH:(k + 1) * GH].double() @ w_ih[k, :, CI:].double()) * slope[:, k * D_:(k + 1) * D_]
                        for k in range(K_)])
    ref_cs = bc0.double() + prod.sum(1)
    errs, cerrs = {}, {}
    for _, mode, _ in MODES:
        kw = dict(A=None, lda=K_ * GH, B=P(w_ih) + 4 * CI, ldb=IN, sB=GH * IN, C=None, ldc=K_ * D_, sC=D_, batch=K_,
                  epi=EPI_LRELU_BWD, pA=plane(ghi, glo, K_ * GH, GH))
        hi = torch.empty(M, K_ * D_, dtype=torch.bfloat16, device=DEV)
        lo = torch.empty_like(hi)
        bc = bc0.clone()
        gemm(mode, 0, 0, M, D_, GH, pOut=plane(hi, lo, K_ * D_, D_), auxp=P(ahi), ldauxp=K_ * D_, sAuxp=D_, colsum=P(bc),
             sColsum=D_, **kw)
        errs[mode] = tile_err(pv(hi, lo).view(M, K_, D_).permute(1, 0, 2), prod)
        cerrs[mode] = max(rel_err(bc[k], ref_cs[k]) for k in range(K_))
        # the fp32 `aux` path given the hi plane's values computes the same bits
        aux = ahi.float()
        hi2, lo2 = torch.empty_like(hi), torch.empty_like(lo)
        gemm(mode, 0, 0, M, D_, GH, pOut=plane(hi2, lo2, K_ * D_, D_), aux=P(aux), ldaux=K_ * D_, sAux=D_, **kw)
        assert same_bits(hi, hi2) and same_bits(lo, lo2), "auxp and aux disagree"
        del hi, lo, hi2, lo2, aux
    check_modes(errs, "cond backward dC M=%d" % M)
    check_modes(cerrs, "cond backward d b_c M=%d" % M)


def test_colsum_with_accumulate_is_refused():
    """With ACCUM the old C would enter the column sums of an unsplit launch but not of a split-K one: refused up front."""
    M, N, Kd = 512, 128, 256
    g = gen(14)
    A, Bm, Cm, cs = randn(Kd, M, g=g), randn(Kd, N, g=g), randn(M, N, g=g), torch.zeros(N, device=DEV)
    L = kp.lib()
    a = kp.GemmArgs(transA=1, transB=0, M=M, N=N, K=Kd, A=P(A), lda=M, B=P(Bm), ldb=N, C=P(Cm), ldc=N, batch=1, epi=EPI_ACCUM,
                    colsum=P(cs))
    ws = torch.empty(int(L.lfi_probe_gemm_ws_bytes(BF16X3, C.byref(a))), dtype=torch.uint8, device=DEV)
    assert L.lfi_probe_gemm(BF16X3, C.byref(a), ws.data_ptr(), ws.numel(), stream()) != 0
    from lets_face_it_b200 import _cabi
    assert b"column sums" in _cabi.lib().lfi_last_error()


# ---- sampler: ACCUM_PRE | LRELU into fp32 C and planes --------------------------------------------------------------
@pytest.mark.parametrize("R", [1024, 200])  # CTA-pair and single-CTA paths
def test_sampler_accum_pre_lrelu(R):
    N = K_ * D_
    g = gen(4)
    A = randn(R, FAR, g=g)
    W = randn(N, FAR, g=g, scale=FAR ** -0.5)
    whi, wlo = planes(W)
    C0 = randn(R, N, g=g)
    ref = lrelu(C0.double() + A.double() @ W.double().T)
    errs, perrs = {}, {}
    for _, mode, _ in MODES:
        Cm = C0.clone()
        hi = torch.empty(R, N, dtype=torch.bfloat16, device=DEV)
        lo = torch.empty_like(hi)
        gemm(mode, 0, 1, R, N, FAR, A=P(A), lda=FAR, B=None, ldb=FAR, C=P(Cm), ldc=N, epi=kp.EPI_ACCUM_PRE | EPI_LRELU,
             pB=plane(whi, wlo, FAR), pOut=plane(hi, lo, N))
        errs[mode] = tile_err(Cm, ref)
        perrs[mode] = tile_err(pv(hi, lo), ref)
        assert same_bits(hi, Cm.to(torch.bfloat16)) and same_bits(lo, (Cm - hi.float()).to(torch.bfloat16))
    check_modes(errs, "sampler C R=%d" % R)
    check_modes(perrs, "sampler planes R=%d" % R)


# ---- flow-step weight gradients: tA = 1, tB = 0, ACCUM, MN-major planes, batch K ----------------------------------------
@pytest.mark.parametrize("B", BATCHES)
def test_flow_weight_gradients(B):
    M = B * TP
    g = gen(5)
    # dW_hh[k] += dA_h[k]^T h[k]: 48 output tiles over a 14,336 / 5,600-row reduction -> split-K
    dAh = randn(K_, M, GH, g=g)
    h = torch.tanh(randn(K_, M, H_, g=g))
    dhi, dlo = planes(dAh)
    hhi, hlo = planes(h)
    C0 = randn(K_, GH, H_, g=g, scale=0.1)
    ref = C0.double() + dAh.double().transpose(1, 2) @ h.double()
    errs = {}
    for _, mode, _ in MODES:
        Cm = C0.clone()
        gemm(mode, 1, 0, GH, H_, M, A=None, lda=GH, B=None, ldb=H_, C=P(Cm), ldc=H_, sC=GH * H_, epi=EPI_ACCUM, batch=K_,
             pA=plane(dhi, dlo, GH, M * GH), pB=plane(hhi, hlo, H_, M * H_))
        errs[mode] = tile_err(Cm, ref)
    check_modes(errs, "dW_hh M=%d" % M, K=M)
    del dAh, h, dhi, dlo, hhi, hlo
    # dW_ih[:, Ci:] += dG^T Cact: column slices of both planes, C at a column offset of [K][GH][In]
    dG = randn(M, K_ * GH, g=g)
    cact = randn(M, K_ * D_, g=g)
    ghi, glo = planes(dG)
    chi, clo = planes(cact)
    W0 = randn(K_, GH, IN, g=g, scale=0.1)
    ref = W0[:, :, CI:].double() + torch.stack([dG[:, k * GH:(k + 1) * GH].double().T @ cact[:, k * D_:(k + 1) * D_].double()
                                               for k in range(K_)])
    errs = {}
    for _, mode, _ in MODES:
        Wm = W0.clone()
        gemm(mode, 1, 0, GH, D_, M, A=None, lda=K_ * GH, B=None, ldb=K_ * D_, C=P(Wm) + 4 * CI, ldc=IN, sC=GH * IN, epi=EPI_ACCUM,
             batch=K_, pA=plane(ghi, glo, K_ * GH, GH), pB=plane(chi, clo, K_ * D_, D_))
        errs[mode] = tile_err(Wm[:, :, CI:], ref)
        assert same_bits(Wm[:, :, :CI], W0[:, :, :CI]), "columns outside the output slice written"
    check_modes(errs, "dW_ih[:, Ci:] M=%d" % M, K=M)


# ---- encoder weight gradients and the dh product ------------------------------------------------------------------
@pytest.mark.parametrize("E,hist,dim", [(128, 2, 30), (256, 16, 30)])
@pytest.mark.parametrize("B", BATCHES)
def test_encoder_weight_gradients_and_dh(E, hist, dim, B):
    M = B * TP
    dimp = (dim + 7) // 8 * 8
    g = gen(6)
    dah = randn(hist * M, 3 * E, g=g)
    dan = randn(hist * M, E, g=g)
    xg = randn(hist * M, dim, g=g)
    hs = torch.tanh(randn(hist * M, E, g=g))
    w_hh = randn(3 * E, E, g=g, scale=E ** -0.5)
    ahi, alo = planes(dah)
    nhi, nlo = planes(dan)
    xhi, xlo = planes(xg, dimp)
    hhi, hlo = planes(hs)
    whi, wlo = planes(w_hh)
    # dW_ih rows [0, 2E) += dA_h[:, :2E]^T x, rows [2E, 3E) += dA_n^T x: N = 30 -> scalar epilogue, split-K atomics
    G0 = randn(3 * E, dim, g=g, scale=0.1)
    ref = G0.double().clone()
    ref[:2 * E] += dah[:, :2 * E].double().T @ xg.double()
    ref[2 * E:] += dan.double().T @ xg.double()
    errs, uerrs, herrs, derrs = {}, {}, {}, {}
    for _, mode, _ in MODES:
        Gm = G0.clone()
        gemm(mode, 1, 0, 2 * E, dim, hist * M, A=None, lda=3 * E, B=None, ldb=dim, C=P(Gm), ldc=dim, epi=EPI_ACCUM,
             pA=plane(ahi, alo, 3 * E), pB=plane(xhi, xlo, dimp))
        gemm(mode, 1, 0, E, dim, hist * M, A=None, lda=E, B=None, ldb=dim, C=P(Gm) + 4 * 2 * E * dim, ldc=dim, epi=EPI_ACCUM,
             pA=plane(nhi, nlo, E), pB=plane(xhi, xlo, dimp))
        errs[mode] = tile_err(Gm, ref)
        # unaligned C base and odd pitch (the scalar path again, reached through the pointer instead of N)
        buf = torch.full((1 + 2 * E * (dim + 1),), float("nan"), device=DEV)
        Cu = buf[1:].view(2 * E, dim + 1)
        Cu[:, :dim] = G0[:2 * E]
        gemm(mode, 1, 0, 2 * E, dim, hist * M, A=None, lda=3 * E, B=None, ldb=dim, C=P(buf) + 4, ldc=dim + 1, epi=EPI_ACCUM,
             pA=plane(ahi, alo, 3 * E), pB=plane(xhi, xlo, dimp))
        uerrs[mode] = tile_err(Cu[:, :dim], ref[:2 * E])
        assert torch.isnan(buf[0]) and torch.isnan(Cu[:, dim]).all(), "unaligned C: pad elements written"
        if hist > 1:  # dW_hh += sum_{s >= 1} dA_h[s]^T h[s-1]
            H0 = randn(3 * E, E, g=g, scale=0.1)
            href = H0.double() + dah[M:].double().T @ hs[:(hist - 1) * M].double()
            Hm = H0.clone()
            gemm(mode, 1, 0, 3 * E, E, (hist - 1) * M, A=None, lda=3 * E, B=None, ldb=E, C=P(Hm), ldc=E, epi=EPI_ACCUM,
                 pA=plane(ahi, alo, 3 * E, off=M * 3 * E), pB=plane(hhi, hlo, E))
            herrs[mode] = tile_err(Hm, href)
        # dh_{s-1} += dA_h W_hh
        dh0 = randn(M, E, g=g)
        dref = dh0.double() + dah[:M].double() @ w_hh.double()
        dhm = dh0.clone()
        gemm(mode, 0, 0, M, E, 3 * E, A=None, lda=3 * E, B=None, ldb=E, C=P(dhm), ldc=E, epi=EPI_ACCUM,
             pA=plane(ahi, alo, 3 * E), pB=plane(whi, wlo, E))
        derrs[mode] = tile_err(dhm, dref)
    check_modes(errs, "encoder dW_ih E=%d hist=%d M=%d" % (E, hist, M), K=hist * M)
    check_modes(uerrs, "encoder dW_ih unaligned C E=%d hist=%d M=%d" % (E, hist, M), K=hist * M)
    if herrs:
        check_modes(herrs, "encoder dW_hh E=%d hist=%d M=%d" % (E, hist, M), K=(hist - 1) * M)
    check_modes(derrs, "encoder dh E=%d M=%d" % (E, M))


# ---- fused encoder-GRU step, enc_gate_fwd ---------------------------------------------------------------------------
class GruCase:
    """Operands of one window step s of an encoder GRU over M = B * T' windows (window m = t' * B + b reads raw frame
    t0 + t' - hist + 1 + s of sequence b)."""

    def __init__(self, E, hist, dim, B, seed):
        g = gen(seed)
        self.E, self.hist, self.dim, self.B, self.M = E, hist, dim, B, B * TP
        self.dimp = (dim + 7) // 8 * 8
        self.x = randn(B, T_, dim, g=g)
        self.w_ih = randn(3 * E, dim, g=g, scale=dim ** -0.5)
        self.w_hh = randn(3 * E, E, g=g, scale=E ** -0.5)
        self.b_ih = randn(3 * E, g=g, scale=0.3)
        self.b_hh = randn(3 * E, g=g, scale=0.3)
        keep = (torch.rand(self.M, hist, generator=g, device=DEV) > 0.4).float()
        self.mask = (keep / 0.6).contiguous()  # frame dropout with p = 0.4, scaled as nn.Dropout
        self.hprev = torch.tanh(randn(self.M, E, g=g))
        self.xp = (self.x.reshape(B * T_, dim) @ self.w_ih.T).contiguous()  # [B*T][3E], row b * T + tau
        self.whi, self.wlo = planes(self.w_hh)
        self.hphi, self.hplo = planes(self.hprev)
        self.wihi, self.wilo = planes(self.w_ih, self.dimp)
        m = torch.arange(self.M, device=DEV)
        self.b_of, self.tp_of = m % B, m // B

    def frames(self, s):
        return T0 + self.tp_of - self.hist + 1 + s

    def xwin(self, s):
        """masked window inputs of step s [M, dim] (fp32, as the library gathers them)"""
        return (self.x[self.b_of, self.frames(s)] * self.mask[:, s:s + 1]).contiguous()

    def ref(self, s, xpath, first):
        E = self.E
        if xpath:  # input projection from the masked window inputs
            ai = self.xwin(s).double() @ self.w_ih.double().T + self.b_ih.double()
        else:
            ai = self.mask[:, s:s + 1].double() * self.xp[self.b_of * T_ + self.frames(s)].double() + self.b_ih.double()
        hp = torch.zeros(self.M, E, dtype=torch.float64, device=DEV) if first else self.hprev.double()
        ah = hp @ self.w_hh.double().T + self.b_hh.double()
        r = torch.sigmoid(ai[:, :E] + ah[:, :E])
        u = torch.sigmoid(ai[:, E:2 * E] + ah[:, E:2 * E])
        n = torch.tanh(ai[:, 2 * E:] + r * ah[:, 2 * E:])
        h = n + u * (hp - n)
        pre = torch.cat([ai[:, :2 * E] + ah[:, :2 * E], ai[:, 2 * E:] + r * ah[:, 2 * E:]], 1)
        return h, torch.cat([r, u, n], 1), ah[:, 2 * E:], pre


def _outs(c, gates16):
    M, E = c.M, c.E
    o = dict(h=torch.empty(M, E, device=DEV), ahn=torch.empty(M, E, device=DEV),
             cond=torch.full((M, FE), float("nan"), device=DEV),
             h_hi=torch.empty(M, E, dtype=torch.bfloat16, device=DEV), h_lo=torch.empty(M, E, dtype=torch.bfloat16, device=DEV))
    o["gates"] = torch.empty(M, 3 * E, dtype=torch.int16 if gates16 else torch.float32, device=DEV)
    return o


def _fused_step(c, mode, s, fuse, gates16, cond_off):
    E, M = c.E, c.M
    o = _outs(c, gates16)
    xa = None
    gru = kp.GruEpi(E=E, s=s, hist=c.hist, B=c.B, T=T_, t0=T0, gates16=gates16, xp=P(c.xp), b_ih=P(c.b_ih), b_hh=P(c.b_hh),
                    mask=P(c.mask), hprev=None if (fuse == kp.FUSE_GRU_FWD_X and s == 0) else P(c.hprev),
                    h=P(o["h"]), gates=P(o["gates"]), ahn=P(o["ahn"]), cond=P(o["cond"]) + 4 * cond_off, cond_ld=FE,
                    h_hi=P(o["h_hi"]), h_lo=P(o["h_lo"]))
    if fuse == kp.FUSE_GRU_FWD_X:
        xa = planes(c.xwin(s), c.dimp)
        gru.xa_hi, gru.xa_lo, gru.xb_hi, gru.xb_lo = P(xa[0]), P(xa[1]), P(c.wihi), P(c.wilo)
        gru.xa_ld = gru.xb_ld = gru.xk = c.dimp
        gru.x_only = 1 if s == 0 else 0
    gemm(mode, 0, 1, M, 3 * E, E, A=None, lda=E, B=None, ldb=E, C=None, ldc=3 * E, pA=plane(c.hphi, c.hplo, E),
         pB=plane(c.whi, c.wlo, E), fuse=fuse, gru=gru)
    return o


def _check_step(c, o, ref, tol, gemm_tol, cond_off, what, pre_scaled=False):
    """pre_scaled: h / gate errors relative to the pre-activations' max|a| per tile (bf16 mode, see the module docstring)"""
    h_ref, g_ref, ahn_ref, pre = ref
    E = c.E
    amax = pre.abs().amax(1, keepdim=True) if pre_scaled else None
    errs = dict(h=tile_err(o["h"], h_ref, None if amax is None else amax.expand(-1, E)), ahn=tile_err(o["ahn"], ahn_ref))
    if o["gates"].dtype == torch.float32:
        errs["gates"] = tile_err(o["gates"], g_ref, None if amax is None else amax.expand(-1, 3 * E))
    assert errs["h"] < tol and errs.get("gates", 0.0) < tol, (what, errs)
    assert errs["ahn"] < gemm_tol, (what, errs)
    # cond: the same bits as h in its column slice, nothing else written
    assert same_bits(o["cond"][:, cond_off:cond_off + E], o["h"]), what
    rest = torch.cat([o["cond"][:, :cond_off], o["cond"][:, cond_off + E:]], 1)
    assert torch.isnan(rest).all(), (what, "cond written outside its slice")
    # h planes: the exact split of the kernel's own h
    assert same_bits(o["h_hi"], o["h"].to(torch.bfloat16)), what
    assert same_bits(o["h_lo"], (o["h"] - o["h_hi"].float()).to(torch.bfloat16)), what
    return errs


def _check_gates16(o16, o32, what):
    """16-bit stash: round(clamp(g) * 65535) for r, u and round(clamp(n) * 32767) for n, off by at most one code."""
    E = o32["h"].shape[1]
    g = o32["gates"].double()
    want_ru = torch.round(g[:, :2 * E].clamp(0, 1) * 65535)
    want_n = torch.round(g[:, 2 * E:].clamp(-1, 1) * 32767)
    got_ru = (o16["gates"][:, :2 * E].int() & 0xFFFF).double()
    got_n = o16["gates"][:, 2 * E:].double()
    d = max(float((got_ru - want_ru).abs().max()), float((got_n - want_n).abs().max()))
    assert d <= 1, (what, "gates16 off by %g codes" % d)
    assert same_bits(o16["h"], o32["h"]), (what, "gates16 changes h")


@pytest.mark.parametrize("E,hist,dim", [(256, 24, 56), (128, 2, 30)])
@pytest.mark.parametrize("B", BATCHES)
def test_fused_gru_step_and_enc_gate_fwd(E, hist, dim, B):
    c = GruCase(E, hist, dim, B, seed=7)
    s1 = hist - 1
    ref_fwd = c.ref(s1, xpath=False, first=False)
    worst = {}
    for name, mode, gemm_tol in MODES:
        tol = STEP_TOL[mode]
        for fuse, s in ((kp.FUSE_GRU_FWD, s1), (kp.FUSE_GRU_FWD_X, 0), (kp.FUSE_GRU_FWD_X, s1)):
            ref = ref_fwd if fuse == kp.FUSE_GRU_FWD else c.ref(s, xpath=True, first=(s == 0))
            for cond_off in (536, 537):  # 16-byte aligned cond slice (128-bit stores) and a misaligned one
                what = "%s fuse=%d s=%d E=%d M=%d cond_off=%d" % (name, fuse, s, E, c.M, cond_off)
                o32 = _fused_step(c, mode, s, fuse, 0, cond_off)
                errs = _check_step(c, o32, ref, tol, gemm_tol, cond_off, what, pre_scaled=(mode == BF16))
                for k, v in errs.items():
                    worst[(name, k)] = max(worst.get((name, k), 0.0), v)
                if cond_off == 536:
                    o16 = _fused_step(c, mode, s, fuse, 1, cond_off)
                    _check_step(c, o16, ref, tol, gemm_tol, cond_off, what + " gates16", pre_scaled=(mode == BF16))
                    _check_gates16(o16, o32, what)
    print("fused GRU step E=%d M=%d" % (E, c.M), {k: "%.2e" % v for k, v in worst.items()})

    # aux::enc_gate_fwd on the same inputs, with the recurrent product given in fp32
    gh = (c.hprev.double() @ c.w_hh.double().T).float().contiguous()
    for gates16 in (0, 1):
        o = _outs(c, gates16)
        a = kp.EncStep(xp=P(c.xp), gh=P(gh), b_ih=P(c.b_ih), b_hh=P(c.b_hh), mask=P(c.mask), hprev=P(c.hprev), h=P(o["h"]),
                       gates=P(o["gates"]), ahn=P(o["ahn"]), cond=P(o["cond"]) + 4 * 536, cond_ld=FE, h_hi=P(o["h_hi"]),
                       h_lo=P(o["h_lo"]), s=s1, hist=hist, B=c.B, T=T_, Tp=TP, t0=T0, E=E, gates16=gates16)
        kp.check(kp.lib().lfi_probe_enc_gate_fwd(C.byref(a), stream()), "enc_gate_fwd")
        torch.cuda.synchronize()
        errs = _check_step(c, o, ref_fwd, EXACT_TOL, EXACT_TOL, 536, "enc_gate_fwd gates16=%d" % gates16)
        if gates16:
            _check_gates16(o, o32_gate, "enc_gate_fwd")
        else:
            o32_gate = o
            print("enc_gate_fwd E=%d M=%d" % (E, c.M), {k: "%.2e" % v for k, v in errs.items()})
    # the bf16x3 fused step agrees with enc_gate_fwd within the GRU bound
    o = _fused_step(c, BF16X3, s1, kp.FUSE_GRU_FWD, 0, 536)
    assert rel_err(o["h"], o32_gate["h"].double()) < GRU_TOL[BF16X3]


# ---- enc_gate_bwd2 ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E", [256, 128])
@pytest.mark.parametrize("B", BATCHES)
def test_enc_gate_bwd2(E, B):
    M = B * TP
    g = gen(8)
    qr = torch.randint(1, 65535, (M, 2 * E), generator=g, device=DEV)
    qn = torch.randint(-32766, 32767, (M, E), generator=g, device=DEV)
    codes = torch.cat([torch.where(qr > 32767, qr - 65536, qr).to(torch.int16), qn.to(torch.int16)], 1).contiguous()
    # the gate values the kernel dequantises (fp32 multiply by the fp32 reciprocal), also fed as the fp32 stash
    gates = torch.cat([qr.float() * torch.tensor(1.0 / 65535, dtype=torch.float32), qn.float() * torch.tensor(1.0 / 32767, dtype=torch.float32)], 1).contiguous()
    ahn = randn(M, E, g=g)
    hprev = torch.tanh(randn(M, E, g=g))
    dh0 = randn(M, E, g=g)
    dcond = randn(M, FE, g=g)
    gbi0, gbh0 = randn(3 * E, g=g, scale=0.01), randn(3 * E, g=g, scale=0.01)
    # fp64 autograd of the GRU cell at the pre-activations that produce these gates
    gd = gates.double()
    ar = torch.logit(gd[:, :E]).requires_grad_()
    au = torch.logit(gd[:, E:2 * E]).requires_grad_()
    ahl = ahn.double().requires_grad_()
    ain = (torch.atanh(gd[:, 2 * E:]) - gd[:, :E] * ahn.double()).requires_grad_()
    hp = hprev.double().requires_grad_()
    r, u = torch.sigmoid(ar), torch.sigmoid(au)
    n = torch.tanh(ain + r * ahl)
    h = n + u * (hp - n)
    dL = dh0.double() + dcond[:, 536:536 + E].double()
    gar, gau, gain, gahn, ghp = torch.autograd.grad(h, [ar, au, ain, ahl, hp], dL)
    dah_ref = torch.cat([gar, gau, gahn], 1)
    terms_ih = torch.cat([gar, gau, gain], 1)
    for gates16 in (0, 1):
        what = "enc_gate_bwd2 E=%d M=%d gates16=%d" % (E, M, gates16)
        dh = dh0.clone()
        dah32, dan32 = torch.empty(M, 3 * E, device=DEV), torch.empty(M, E, device=DEV)
        dah_hi, dah_lo = torch.empty(M, 3 * E, dtype=torch.bfloat16, device=DEV), torch.empty(M, 3 * E, dtype=torch.bfloat16, device=DEV)
        dan_hi, dan_lo = torch.empty(M, E, dtype=torch.bfloat16, device=DEV), torch.empty(M, E, dtype=torch.bfloat16, device=DEV)
        gbi, gbh = gbi0.clone(), gbh0.clone()
        a = kp.EncStepBwd2(gates=P(codes if gates16 else gates), ahn=P(ahn), hprev=P(hprev), dh=P(dh), dh_extra=P(dcond) + 4 * 536,
                           dh_extra_ld=FE, dah32=P(dah32), dan32=P(dan32), dah_hi=P(dah_hi), dah_lo=P(dah_lo), dan_hi=P(dan_hi),
                           dan_lo=P(dan_lo), gb_ih=P(gbi), gb_hh=P(gbh), M=M, E=E, gates16=gates16)
        kp.check(kp.lib().lfi_probe_enc_gate_bwd2(C.byref(a), stream()), "enc_gate_bwd2")
        torch.cuda.synchronize()
        errs = dict(dah=tile_err(dah32, dah_ref), dan=tile_err(dan32, gain), dh=tile_err(dh, ghp))
        errs["gb_ih"] = sum_err(gbi, gbi0.double() + terms_ih.sum(0), terms_ih.abs().sum(0))
        errs["gb_hh"] = sum_err(gbh, gbh0.double() + dah_ref.sum(0), dah_ref.abs().sum(0))
        assert errs["dah"] < EXACT_TOL and errs["dan"] < EXACT_TOL and errs["dh"] < EXACT_TOL, (what, errs)
        assert errs["gb_ih"] < SUM_TOL and errs["gb_hh"] < SUM_TOL, (what, errs)
        for hi, lo, v in ((dah_hi, dah_lo, dah32), (dan_hi, dan_lo, dan32)):
            assert same_bits(hi, v.to(torch.bfloat16)) and same_bits(lo, (v - hi.float()).to(torch.bfloat16)), what
        print(what, {k: "%.2e" % v for k, v in errs.items()})


# ---- colsum_planes: the two bias-gradient reductions of the tensor-core backward pipeline ----------------------------
@pytest.mark.parametrize("B", BATCHES)
def test_colsum_planes(B):
    M = B * TP
    g = gen(9)
    dG = randn(M, K_ * GH, g=g)
    dAh = randn(K_, M, GH, g=g)
    for name, mode, _ in MODES:
        ghi, glo = planes(dG)
        ahi, alo = planes(dAh)
        if mode == BF16:
            glo = alo = None
        gv = ghi.double() + (glo.double() if glo is not None else 0)
        av = ahi.double() + (alo.double() if alo is not None else 0)
        b_ih0, b_hh0 = randn(K_ * GH, g=g, scale=0.1), randn(K_ * GH, g=g, scale=0.1)
        b_ih, b_hh = b_ih0.clone(), b_hh0.clone()
        L = kp.lib()
        # d b_ih = colsum(dG) over all K slices; its r, u parts (j % GH < 2H) are d b_hh's too
        kp.check(L.lfi_probe_colsum_planes(P(b_ih), P(b_hh), GH, 2 * H_, 0, P(ghi), P(glo), K_ * GH, 0, 1, M, 0, K_ * GH, stream()), "colsum_planes")
        torch.cuda.synchronize()
        ru = (torch.arange(K_ * GH, device=DEV) % GH) < 2 * H_
        cs, ab = gv.sum(0), gv.abs().sum(0)
        e1 = sum_err(b_ih, b_ih0.double() + cs, ab)
        e2 = sum_err(b_hh[ru], b_hh0[ru].double() + cs[ru], ab[ru])
        assert same_bits(b_hh[~ru], b_hh0[~ru]), "out2 written outside j % period < lim2"
        # d b_hh n part += colsum of the n columns of dA_h, batched over K with the output stride GH
        b2 = b_hh.clone()
        kp.check(L.lfi_probe_colsum_planes(P(b_hh) + 4 * 2 * H_, None, 1, 0, GH, P(ahi), P(alo), GH, M * GH, K_, M, 2 * H_, H_, stream()),
                 "colsum_planes")
        torch.cuda.synchronize()
        want = b2.double().view(K_, GH).clone()
        want[:, 2 * H_:] += av[:, :, 2 * H_:].sum(1)
        e3 = sum_err(b_hh.view(K_, GH)[:, 2 * H_:], want[:, 2 * H_:], av[:, :, 2 * H_:].abs().sum(1))
        assert same_bits(b_hh.view(K_, GH)[:, :2 * H_], b2.view(K_, GH)[:, :2 * H_])
        assert max(e1, e2, e3) < SUM_TOL, (name, e1, e2, e3)
        print("colsum_planes %s M=%d: %.2e %.2e %.2e" % (name, M, e1, e2, e3))


# ---- split_to_planes / gather_windows_planes: bit-exact against torch's round-to-nearest-even -----------------------------
def test_split_to_planes_bit_exact():
    g = gen(10)
    L = kp.lib()
    cases = [  # src, rows, cols, ld, stride, batch, offset (floats)
        (randn(3 * 128, 30, g=g), 3 * 128, 30, 30, 0, 1, 0),                   # W_ih of a speech encoder: pitch 32
        (randn(K_, GH, IN, g=g), GH, D_, IN, GH * IN, K_, CI),                # gate-ih weight columns [Ci, In), batch K
        (randn(K_ * D_, FE, g=g), K_ * D_, FAR, FE, 0, 1, 0),                 # the sampler's p1_face part of WcF
        (randn(777, 61, g=g), 777, 61, 61, 0, 1, 0),                           # odd width, odd pitch (scalar loads)
    ]
    for src, rows, cols, ld, stride, batch, off in cases:
        ldp = (cols + 7) // 8 * 8
        hi = torch.full((batch, rows, ldp), 0x7F7F, dtype=torch.int16, device=DEV).view(torch.bfloat16)
        lo = hi.clone()
        kp.check(L.lfi_probe_split_to_planes(P(src) + 4 * off, rows, cols, ld, stride, batch, P(hi), P(lo), stream()), "split_to_planes")
        torch.cuda.synchronize()
        v = torch.as_strided(src, (batch, rows, cols), (stride or rows * ld, ld, 1), storage_offset=off)
        whi, wlo = planes(v, ldp)
        assert same_bits(hi, whi) and same_bits(lo, wlo), (rows, cols, ld, batch)
        assert not bits(hi[..., cols:]).any() and not bits(lo[..., cols:]).any(), "padding columns must be zero"


@pytest.mark.parametrize("B", BATCHES)
def test_gather_windows_planes_bit_exact(B):
    g = gen(11)
    L = kp.lib()
    for E, hist, dim in ENCODERS:
        c = GruCase(E, hist, dim, B, seed=12)
        ldp = c.dimp
        hi = torch.full((hist, c.M, ldp), 0x7F7F, dtype=torch.int16, device=DEV).view(torch.bfloat16)
        lo = hi.clone()
        kp.check(L.lfi_probe_gather_windows_planes(P(hi), P(lo), ldp, P(c.x), P(c.mask), B, T_, dim, hist, 1, T0, TP, stream()),
                 "gather_windows_planes")
        torch.cuda.synchronize()
        for s in range(hist):
            whi, wlo = planes(c.xwin(s), ldp)
            assert same_bits(hi[s], whi) and same_bits(lo[s], wlo), (E, hist, dim, s)
        assert not bits(hi[..., dim:]).any() and not bits(lo[..., dim:]).any()


# ---- persistent window-GRU forward ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("E,hist,dim", ENCODERS)
@pytest.mark.parametrize("B", BATCHES)
def test_persistent_encoder_forward(E, hist, dim, B):
    c = GruCase(E, hist, dim, B, seed=13)
    L = kp.lib()
    M = c.M
    # time-major raw-frame projections (row r = tau * B + b), row-interleaved, rows padded to 32 (enc_persist.cuh)
    xp_tm = c.x.permute(1, 0, 2).reshape(T_ * B, dim) @ c.w_ih.T
    R = (T_ * B + 31) // 32 * 32
    xp_tiled = F.pad(xp_tm, (0, 0, 0, R - T_ * B)).view(R // 32, 32, 3 * E // 4, 4).permute(0, 2, 1, 3).contiguous()
    # fp64 reference: the window GRU from a zero state over all hist steps
    h = torch.zeros(M, E, dtype=torch.float64, device=DEV)
    for s in range(hist):
        ai = c.mask[:, s:s + 1].double() * xp_tm[c.frames(s) * B + c.b_of].double() + c.b_ih.double()
        ah = h @ c.w_hh.double().T + c.b_hh.double()
        r = torch.sigmoid(ai[:, :E] + ah[:, :E])
        u = torch.sigmoid(ai[:, E:2 * E] + ah[:, E:2 * E])
        n = torch.tanh(ai[:, 2 * E:] + r * ah[:, 2 * E:])
        h = n + u * (h - n)
    for name, mode, _ in MODES:
        assert L.lfi_probe_enc_fwd_supported(E, hist, M, mode) == 1
        cond = torch.full((M, FE), float("nan"), device=DEV)
        a = kp.FwdArgs(E=E, hist=hist, B=B, T=T_, t0=T0, M=M, nplanes=2 if mode == BF16X3 else 1, xp=P(xp_tiled), b_ih=P(c.b_ih),
                       b_hh=P(c.b_hh), mask=P(c.mask), whh_hi=P(c.whi), whh_lo=P(c.wlo), cond=P(cond) + 4 * 536, cond_ld=FE)
        kp.check(L.lfi_probe_enc_launch_fwd(C.byref(a), stream()), "encp::launch_fwd")
        torch.cuda.synchronize()
        err = tile_err(cond[:, 536:536 + E], h)
        rest = torch.cat([cond[:, :536], cond[:, 536 + E:]], 1)
        assert torch.isnan(rest).all(), "cond written outside its slice"
        assert err < GRU_TOL[mode], (name, E, hist, M, err)
        print("persistent encoder %s E=%d hist=%d M=%d: %.2e" % (name, E, hist, M, err))
