"""CPU: the test-only probe library (tests/csrc/kernel_probe.cu) loads next to liblfi_b200.so, exports every wrapper
tests/test_gpu_kernel_units.py binds, and the ctypes mirrors of the internal argument structs match the compiler's layout
(a field out of place would silently hand a kernel the wrong pointer)."""
import ctypes
import os

from tests import kernel_probe as kp


def test_probe_exports_every_bound_wrapper():
    lib = kp.lib()
    for name in kp.SIGNATURES:
        assert hasattr(lib, name), "missing export %s" % name


def test_probe_resolves_against_the_package_library():
    from lets_face_it_b200 import _cabi

    kp.lib()
    # the probe's internal symbols come from the already loaded package library, not from a second copy
    maps = open("/proc/self/maps").read()
    libs = {line.split()[-1] for line in maps.splitlines() if line.rstrip().endswith("liblfi_b200.so")}
    assert {os.path.realpath(p) for p in libs} == {os.path.realpath(_cabi.LIB_PATH)}, libs


def test_struct_mirrors_match_the_compiler_layout():
    for st in kp.STRUCTS:
        name = st.__name__
        assert kp.layout(name) == ctypes.sizeof(st), (name, kp.layout(name), ctypes.sizeof(st))
        for fname, _ in st._fields_:
            assert kp.layout(name, fname) == getattr(st, fname).offset, (name, fname, kp.layout(name, fname), getattr(st, fname).offset)
    assert kp.layout("GemmArgs", "no_such_field") == ctypes.c_size_t(-1).value
