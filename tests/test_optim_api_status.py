"""CPU: the fused SGD / RMSprop entry points of ABI 10 (lfi_clip_sgd_dev / lfi_clip_rmsprop_dev) reject every bad argument with
LFI_ERR_ARG before they launch anything (no compute: every call below returns from its argument checks, and the launch counter
does not move)."""
from lets_face_it_b200 import _cabi

LFI_ERR_ARG = -3
FAKE = 1 << 20  # never dereferenced: the checks run first
N = 1000


def _sgd(theta=FAKE, grad=FAKE, buf=FAKE, n=N, hyper=FAKE, momentum=0.9, dampening=0.0, wd=0.0, nesterov=0, scratch=FAKE):
    return _cabi.lib().lfi_clip_sgd_dev(theta, grad, buf, n, hyper, momentum, dampening, wd, nesterov, 20.0, 1.0, scratch, None)


def _rms(theta=FAKE, grad=FAKE, sq=FAKE, ga=FAKE, buf=FAKE, n=N, hyper=FAKE, alpha=0.99, eps=1e-8, wd=0.0, momentum=0.9, scratch=FAKE):
    return _cabi.lib().lfi_clip_rmsprop_dev(theta, grad, sq, ga, buf, n, hyper, alpha, eps, wd, momentum, 20.0, 1.0, scratch, None)


def test_sgd_rejects_arguments():
    L = _cabi.lib()
    n0 = L.lfi_launch_count()
    assert _sgd(theta=None) == LFI_ERR_ARG
    assert _sgd(grad=None) == LFI_ERR_ARG
    assert _sgd(hyper=None) == LFI_ERR_ARG
    assert _sgd(scratch=None) == LFI_ERR_ARG
    assert _sgd(n=0) == LFI_ERR_ARG
    assert _sgd(buf=None) == LFI_ERR_ARG                    # momentum without its buffer
    assert _sgd(momentum=0.0) == LFI_ERR_ARG                # a buffer without momentum
    assert _sgd(momentum=-0.5) == LFI_ERR_ARG
    assert _sgd(wd=-1.0) == LFI_ERR_ARG
    assert _sgd(nesterov=1, momentum=0.0, buf=None) == LFI_ERR_ARG
    assert _sgd(nesterov=1, dampening=0.1) == LFI_ERR_ARG
    assert L.lfi_launch_count() == n0
    assert b"nesterov" in L.lfi_last_error()


def test_rmsprop_rejects_arguments():
    L = _cabi.lib()
    n0 = L.lfi_launch_count()
    assert _rms(theta=None) == LFI_ERR_ARG
    assert _rms(grad=None) == LFI_ERR_ARG
    assert _rms(sq=None) == LFI_ERR_ARG
    assert _rms(hyper=None) == LFI_ERR_ARG
    assert _rms(scratch=None) == LFI_ERR_ARG
    assert _rms(n=0) == LFI_ERR_ARG
    assert _rms(buf=None) == LFI_ERR_ARG                    # momentum without its buffer
    assert _rms(momentum=0.0) == LFI_ERR_ARG                # a buffer without momentum
    assert _rms(momentum=-0.5, buf=None) == LFI_ERR_ARG
    assert _rms(alpha=-0.1) == LFI_ERR_ARG
    assert _rms(eps=-1e-8) == LFI_ERR_ARG
    assert _rms(wd=-1.0) == LFI_ERR_ARG
    assert L.lfi_launch_count() == n0
