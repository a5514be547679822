"""CPU: the shape classes of the MF-Q Ising dispatch, derived from the library, each have a representative in the GPU
tests of tests/test_cuda_ising_shapes.py.

`mfi_resident_cluster_size(dtype, side)` is host-only and the library loads without a GPU, so this runs everywhere the
library is built.  A class is (dtype, kernel, CTAs per lattice C, FAST): kernel is K6r (the generic cluster kernel),
K6s (the persistent fp32 kernel at the sides it is specialised for) or K6 (streaming only: no resident kernel).  FAST
is the generic K6r's compile-time flag: side % 32 == 0 and (side / C) % 4 == 0, every thread owns four live sites and a
row's wrap is a word wrap; otherwise the `x < L` lanes, partial words and per-site halo reads are live.  A dispatch
change that creates a class fails here until the GPU tests cover it."""
import ctypes
import os

import pytest

from conftest import PKG

SO = os.path.join(PKG, "build", "libmagent.so")

F32, F64 = 0, 1
SIDES = range(3, 1025)              # mfi_step accepts sides 3 .. 1024, less what the two limits below refuse
STREAM_MAX = {F32: 896, F64: 512}   # K6: two bit planes of side x ceil(side / 32) words within 200 KB; fp64 up to 512
K6S_SIDES = (64, 128, 256, 512)     # fp32 sides that launch_ising_persistent sends to K6s by default

# ---- the representatives, shared with tests/test_cuda_ising_shapes.py -------------------------------------------
# part 2: every resident / streaming class against the fp64 oracle
FP32_RESIDENT = (3, 31, 32, 33, 63, 72, 80, 96, 112, 160, 192)
FP32_STREAM = (100, 513, 640, 896)
FP64_RESIDENT = (3, 32, 50, 56, 64, 80, 96, 128, 192)
FP64_STREAM = (52, 130)
# part 3: production draws beyond the top bit, (dtype, side) per kernel
DRAW_SIDES = ((F32, 100), (F64, 52),                       # K6
              (F32, 33), (F32, 80), (F32, 192), (F64, 56), (F64, 128),   # generic K6r
              (F32, 64), (F32, 128), (F32, 256), (F32, 512))  # K6s


def representatives():
    """(dtype, side) of every parametrised MF-Q shape in the GPU file"""
    reps = {(F32, L) for L in FP32_RESIDENT + FP32_STREAM} | {(F64, L) for L in FP64_RESIDENT + FP64_STREAM}
    return reps | set(DRAW_SIDES)


def load():
    lib = ctypes.CDLL(SO)
    lib.mfi_resident_cluster_size.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.mfi_resident_cluster_size.restype = ctypes.c_int
    return lib


def shape_class(lib, dtype, side):
    C = lib.mfi_resident_cluster_size(dtype, side)
    if dtype == F32 and side in K6S_SIDES:
        return ("fp32", "K6s", C, None)
    if C == 0:
        return ("fp32" if dtype == F32 else "fp64", "K6", 0, None)
    return ("fp32" if dtype == F32 else "fp64", "K6r", C, side % 32 == 0 and (side // C) % 4 == 0)


def classes(lib):
    """{class: [sides]} over every side 3 .. 1024 that some kernel takes, both dtypes"""
    out = {}
    for dtype in (F32, F64):
        for side in SIDES:
            c = shape_class(lib, dtype, side)
            if c[1] != "K6" or side <= STREAM_MAX[dtype]:       # past STREAM_MAX only a resident kernel would take it
                out.setdefault(c, []).append(side)
    return out


@pytest.mark.skipif(not os.path.exists(SO), reason="library not built")
def test_every_shape_class_has_a_representative(capsys):
    lib = load()
    found = classes(lib)
    reps = representatives()
    covered = {shape_class(lib, d, L) for d, L in reps}
    with capsys.disabled():
        print("\n[ising shape classes] %d classes over sides %d..%d:" % (len(found), SIDES[0], SIDES[-1]))
        for c, sides in sorted(found.items(), key=repr):
            rep = sorted(L for d, L in reps if shape_class(lib, d, L) == c)
            print("  %-36s %4d sides (%d..%d), tested at %s" % (c, len(sides), sides[0], sides[-1], rep))
    missing = {c: sides[:8] for c, sides in found.items() if c not in covered}
    assert not missing, "shape classes without a representative in tests/test_cuda_ising_shapes.py: %r" % missing
    # the K6s sides really are resident (K6s, C = strips per lattice), and every representative is a side mfi_step takes
    assert all(lib.mfi_resident_cluster_size(F32, L) > 0 for L in K6S_SIDES)
    assert all(3 <= L <= STREAM_MAX[d] for d, L in reps)


@pytest.mark.skipif(not os.path.exists(SO), reason="library not built")
@pytest.mark.parametrize("dtype,side", [(F32, STREAM_MAX[F32] + 1), (F64, STREAM_MAX[F64] + 1), (F32, 1025), (F32, 2)])
def test_sides_past_the_streaming_limits_are_refused_before_launch(dtype, side):
    """the upper ends of SIDES as the library has them: mfi_step refuses these sides on the host, before it touches the
    device (so the null pointers are never used), which is what makes STREAM_MAX the last streaming side"""
    lib = load()
    lib.mfi_step.restype = ctypes.c_int
    lib.mfb_last_error.restype = ctypes.c_char_p
    rc = lib.mfi_step(dtype, 1, side, None, None, ctypes.c_double(1.0), ctypes.c_double(0.1), None, None, 0, 0, 0,
                      None, None, None, None)
    assert rc == -1
    msg = lib.mfb_last_error().decode()
    assert msg.startswith("mfi_step: ") and ("side" in msg or "too large" in msg), msg
