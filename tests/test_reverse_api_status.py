"""CPU: the reverse-direction FlowStep entry points of ABI 9 (lfi_flowstep_rev_fwd_train / lfi_flowstep_rev_bwd) reject a null
pointer, a too-small stash or a too-small workspace with a status before they launch anything (no compute: every call below
returns from its argument checks, and the launch counter does not move)."""
import ctypes

from lets_face_it_b200 import _cabi

LFI_ERR_ARG, LFI_ERR_WORKSPACE = -3, -4
FAKE = 1 << 20  # never dereferenced: the checks run first


def _shape(G=3):
    sh = _cabi.Shape()
    sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps, sh.f_raw = 7, 3, 16, 24, G, 1, 1e-4, 40
    return sh


def _params():
    P = _cabi.Params()
    for n in ("an_bias", "an_logs", "w", "wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf"):
        setattr(P, n, FAKE)
    return P


def test_reverse_sizes():
    L = _cabi.lib()
    for G in (3, 4):
        sh = _shape(G)
        assert L.lfi_flowstep_rev_bwd_ws_bytes(ctypes.byref(sh), 21) > 0
        assert L.lfi_flowstep_rev_bwd_ws_bytes(ctypes.byref(sh), 0) == 0


def test_rev_fwd_train_rejects_arguments():
    L = _cabi.lib()
    sh, P, B = _shape(), _params(), 21
    ws = L.lfi_flowstep_ws_bytes(ctypes.byref(sh), B)
    stash = L.lfi_flowstep_stash_bytes(ctypes.byref(sh), B)

    def call(derived, s, sb, w, wb, c_out=None, shape=sh):
        return L.lfi_flowstep_rev_fwd_train(ctypes.byref(shape), derived, ctypes.byref(P), 1, FAKE, FAKE, None, None, FAKE, c_out, FAKE,
                                            FAKE, B, s, sb, w, wb, None)

    n0 = L.lfi_launch_count()
    assert call(None, FAKE, stash, FAKE, ws) == LFI_ERR_ARG
    assert call(FAKE, None, stash, FAKE, ws) == LFI_ERR_ARG
    assert call(FAKE, FAKE, stash, None, ws) == LFI_ERR_ARG
    assert call(FAKE, FAKE, stash - 1, FAKE, ws) == LFI_ERR_WORKSPACE
    assert call(FAKE, FAKE, stash, FAKE, ws - 1) == LFI_ERR_WORKSPACE
    lstm = _shape(4)
    big = 1 << 30
    assert call(FAKE, FAKE, big, FAKE, big, shape=lstm) == LFI_ERR_ARG  # LSTM without c_out
    assert L.lfi_launch_count() == n0


def test_rev_bwd_rejects_arguments():
    L = _cabi.lib()
    sh, P, G, B = _shape(), _params(), _params(), 21
    ws = L.lfi_flowstep_rev_bwd_ws_bytes(ctypes.byref(sh), B)
    stash = L.lfi_flowstep_stash_bytes(ctypes.byref(sh), B)

    def call(s, sb, w, wb, dx=FAKE, g=G):
        return L.lfi_flowstep_rev_bwd(ctypes.byref(sh), FAKE, ctypes.byref(P), 1, FAKE, None, None, FAKE, None, None, None, dx, FAKE, FAKE,
                                      None, ctypes.byref(g), B, s, sb, w, wb, None)

    n0 = L.lfi_launch_count()
    assert call(None, stash, FAKE, ws) == LFI_ERR_ARG
    assert call(FAKE, stash, None, ws) == LFI_ERR_ARG
    assert call(FAKE, stash, FAKE, ws, dx=None) == LFI_ERR_ARG
    no_w = _params()
    no_w.w = None
    assert call(FAKE, stash, FAKE, ws, g=no_w) == LFI_ERR_ARG
    assert call(FAKE, stash - 1, FAKE, ws) == LFI_ERR_WORKSPACE
    assert call(FAKE, stash, FAKE, ws - 1) == LFI_ERR_WORKSPACE
    assert L.lfi_launch_count() == n0
