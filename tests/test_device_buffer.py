"""DeviceBuffer (armour_b200/csrc/device_buffer.h), the owner of every device allocation of the C API's contexts, WITHOUT a GPU.

tests/emu/device_buffer_driver.cpp compiles the header with g++ against stand-ins of cudaMalloc / cudaFree that count the
live allocations, spot frees of pointers that are not live, and can be told to fail.  The failure cases are the point:
after a failed reserve the buffer must be empty (null, capacity 0), so that a later reserve of a size the lost allocation
would have held allocates again instead of handing out a null pointer.
"""
import ctypes as C
import os
import subprocess

import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "emu", "device_buffer_driver.cpp")
CUDA_ERROR_MEMORY_ALLOCATION = 2


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("device_buffer") / "libdevice_buffer_driver.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([cxx, "-O1", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared", "-o", so, SRC], check=True,
                   capture_output=True)
    lib = C.CDLL(so)
    vp, sz = C.c_void_p, C.c_size_t
    for name, res, args in [("buf_new", vp, []), ("buf_delete", None, [vp]), ("buf_reserve", C.c_int, [vp, sz]),
                            ("buf_capacity", sz, [vp]), ("buf_get", vp, [vp]), ("buf_move_new", vp, [vp]),
                            ("buf_move_assign", None, [vp, vp]), ("stub_fail_next", None, [C.c_int]),
                            ("stub_live", C.c_long, []), ("stub_mallocs", C.c_long, []), ("stub_frees", C.c_long, []),
                            ("stub_bad_frees", C.c_long, []), ("stub_last_bytes", sz, [])]:
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib


def counts(lib):
    return dict(live=lib.stub_live(), mallocs=lib.stub_mallocs(), frees=lib.stub_frees(), bad=lib.stub_bad_frees())


def delta(lib, before):
    now = counts(lib)
    return {k: now[k] - before[k] for k in now}


def test_reserve_grows_and_never_shrinks(lib):
    c0 = counts(lib)
    b = lib.buf_new()
    assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0
    assert lib.buf_reserve(b, 10) == 0
    assert lib.buf_capacity(b) == 10 and lib.buf_get(b) is not None and lib.stub_last_bytes() == 80
    assert lib.buf_reserve(b, 4) == 0
    assert lib.buf_capacity(b) == 10  # a smaller request keeps the larger allocation
    assert lib.buf_reserve(b, 25) == 0
    assert lib.buf_capacity(b) == 25 and lib.stub_last_bytes() == 200
    assert delta(lib, c0) == dict(live=1, mallocs=2, frees=1, bad=0)  # the old allocation was freed before the new one
    lib.buf_delete(b)
    assert delta(lib, c0) == dict(live=0, mallocs=2, frees=2, bad=0)


def test_reserve_that_fits_does_not_reallocate(lib):
    b = lib.buf_new()
    assert lib.buf_reserve(b, 16) == 0
    p, c0 = lib.buf_get(b), counts(lib)
    for n in (16, 15, 1, 0):
        assert lib.buf_reserve(b, n) == 0
        assert lib.buf_get(b) == p and lib.buf_capacity(b) == 16
    assert delta(lib, c0) == dict(live=0, mallocs=0, frees=0, bad=0)
    lib.buf_delete(b)


def test_reserve_of_nothing_allocates_nothing(lib):
    c0 = counts(lib)
    b = lib.buf_new()
    assert lib.buf_reserve(b, 0) == 0
    assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0
    lib.buf_delete(b)
    assert delta(lib, c0) == dict(live=0, mallocs=0, frees=0, bad=0)


def test_failed_reserve_leaves_an_empty_buffer(lib):
    b = lib.buf_new()
    assert lib.buf_reserve(b, 100) == 0
    c0 = counts(lib)
    lib.stub_fail_next(1)
    assert lib.buf_reserve(b, 200) == CUDA_ERROR_MEMORY_ALLOCATION
    assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0  # not the old capacity (100) or the requested one (200)
    assert delta(lib, c0) == dict(live=-1, mallocs=0, frees=1, bad=0)  # the old allocation is gone
    # every size allocates again, also one the lost allocation would have held
    for n in (50, 100, 300):
        lib.stub_fail_next(1)
        assert lib.buf_reserve(b, n) == CUDA_ERROR_MEMORY_ALLOCATION
        assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0
        assert lib.buf_reserve(b, n) == 0
        assert lib.buf_get(b) is not None and lib.buf_capacity(b) == n and lib.stub_last_bytes() == 8 * n
    lib.buf_delete(b)
    assert delta(lib, c0) == dict(live=-1, mallocs=3, frees=4, bad=0)


def test_failed_first_reserve(lib):
    c0 = counts(lib)
    b = lib.buf_new()
    lib.stub_fail_next(1)
    assert lib.buf_reserve(b, 8) == CUDA_ERROR_MEMORY_ALLOCATION
    assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0
    lib.buf_delete(b)  # frees nothing: the stand-in's failure value is never taken for an allocation
    assert delta(lib, c0) == dict(live=0, mallocs=0, frees=0, bad=0)


def test_destruction_and_moves_free_exactly_once(lib):
    c0 = counts(lib)
    a = lib.buf_new()
    assert lib.buf_reserve(a, 10) == 0
    pa = lib.buf_get(a)
    b = lib.buf_move_new(a)  # move construction takes the allocation over
    assert lib.buf_get(b) == pa and lib.buf_capacity(b) == 10
    assert lib.buf_get(a) is None and lib.buf_capacity(a) == 0
    lib.buf_delete(a)
    assert delta(lib, c0) == dict(live=1, mallocs=1, frees=0, bad=0)

    c = lib.buf_new()
    assert lib.buf_reserve(c, 4) == 0
    lib.buf_move_assign(c, b)  # move assignment frees c's allocation and takes b's
    assert lib.buf_get(c) == pa and lib.buf_capacity(c) == 10
    assert lib.buf_get(b) is None and lib.buf_capacity(b) == 0
    assert delta(lib, c0) == dict(live=1, mallocs=2, frees=1, bad=0)
    lib.buf_move_assign(c, c)  # self-assignment keeps the allocation
    assert lib.buf_get(c) == pa and lib.buf_capacity(c) == 10
    lib.buf_move_assign(c, b)  # assigning an empty buffer frees
    assert lib.buf_get(c) is None and lib.buf_capacity(c) == 0
    lib.buf_delete(b)
    lib.buf_delete(c)
    assert delta(lib, c0) == dict(live=0, mallocs=2, frees=2, bad=0)
