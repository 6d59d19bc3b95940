"""The generic passes at the extents they actually serve: camera-width axes, large prime factors, the 12800-point limit,
and the AUTO rule that sends a stack to them.

The power-of-two fast path stops at 1024 points per axis, and periodic embedding needs image + kernel - 1 <= 1024 on
every axis (csrc/api.cu, want_embedding / fast_extents).  Every stack with a longer axis -- 2048 x 2048 or 2160 x 2560
sCMOS frames, a 1000-pixel axis with a 41-point PSF -- runs natively on the generic passes (csrc/fft_generic.cuh):
- an axis longer than 1024 points runs with L = 2048 / n = 1 line per block (csrc/engine.cu, build_axis);
- above 3072 points the two shared-memory line buffers, 16 n bytes, exceed the 48 KB default and rely on the
  cudaFuncSetAttribute calls of get_fft_plan, up to kMaxSmem = 200 KB at n = 12800; longer axes are rejected;
- a prime factor p is one direct p-point DFT stage accumulated in float32 (smem_fft): its error grows with p.

Every case asserts its route first (last_geometry() of the one-shot call, the strategy of a handle at those extents),
so that a shape that silently changes route fails here instead of passing while testing other code.  Then it compares
against the oracle with the parity tolerances (tests/parity_cases.py).

The `emu` fixture runs the shared cases in the CPU suite on the host-emulation build; the `gpu` fixture runs them on the
product library, together with the camera-frame deconvolutions.  The routing table and the unbounded-extent rejections
are host logic and run on the emulator only.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.fft as sfft

from libmultiviewnative_b200 import capi
from libmultiviewnative_b200.synthetic import make_views, make_views_fast
from oracle import mvn_oracle as orc
from tests import parity_cases as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
NATIVE, EMBEDDED, ZERO_PADDED = pc.GEOMETRY_NATIVE, pc.GEOMETRY_EMBEDDED, pc.GEOMETRY_ZERO_PADDED
LIMIT_MESSAGE = "exceeds the shared-memory transform limit"
MAX_AXIS = 12800  # kMaxSmem / (2 buffers x 8-byte complex), csrc/engine.cu


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def L(request):
    if request.param == "emu":
        from libmultiviewnative_b200._build import build_emu

        lib = capi.Library(build_emu())
    else:
        lib = capi.load()
        assert "sm_100a" in lib.version()
    yield lib
    lib.release_cached_memory()


@pytest.fixture(scope="module")
def E():
    from libmultiviewnative_b200._build import build_emu

    lib = capi.Library(build_emu())
    yield lib
    lib.release_cached_memory()


@pytest.fixture(scope="module")
def G():
    lib = capi.load()
    assert "sm_100a" in lib.version() and lib.num_devices() >= 1
    yield lib
    lib.release_cached_memory()


def _emulated(L):
    return "emulation" in L.version()


def _strategy(L, dims, kdims=None, geometry="native"):
    with L.plan(dims, 1, max_kernel_dims=kdims, geometry=geometry) as p:
        info = p.info()
        return int(info.strategy), tuple(int(d) for d in info.dims)


def _random_conv(dims, kdims, seed):
    rng = np.random.default_rng(seed)
    img = (rng.random(dims) + 1).astype(F32)
    k = rng.random(kdims).astype(F32)
    k /= k.sum()
    return img, k


def _assert_conv_close(got, exp):
    """the convolution tolerances of tests/parity_cases.py"""
    assert pc.rel_l2(got, exp) <= 1e-5, (pc.max_rel(got, exp), pc.rel_l2(got, exp))
    assert float(np.max(np.abs(got.astype(np.float64) - exp))) <= 1e-4 * float(np.max(np.abs(exp)))


def _f64_convolution(img, k):
    dims = img.shape
    kh = sfft.rfftn(orc.wrap_kernel(k, dims).astype(np.float64))
    return sfft.irfftn(sfft.rfftn(img.astype(np.float64)) * kh, s=dims)


# ---- a. long axes on x, y and z ------------------------------------------------------------------------------------
# length: why
#   1025 = 5^2 41          the first L = 1 length, radix 41
#   1031 (prime)           L = 1, one direct 1031-point stage
#   2048                   a power of two the fast path does not take
#   2160 = 2^4 3^3 5       camera width, radices 3 and 5
#   2560 = 2^9 5           camera width
#   3200 = 2^7 5^2         first case above 48 KB of shared memory (51 200 B)
#   4099 (prime)           > 48 KB, one direct 4099-point stage
#   12800 = 2^9 5^2        exactly kMaxSmem (204 800 B)
#   12799 (prime)          the largest prime the library accepts: the longest float32 accumulation
LONG_AXES = [1025, 1031, 2048, 2160, 2560, 3200, 4099, 12800, 12799]
PRIMES = {1031, 4099, 12799}
EMU_SKIPPED = {4099, 12799}  # O(p^2) stages: hundreds of millions to billions of emulated multiply-adds
SHORT = (4, 6)  # the two other axes
KLONG, KSHORT = 41, 3


def _long_axis_shape(axis, n):
    dims, kdims = list(SHORT), [KSHORT, KSHORT]
    dims.insert(axis, n)
    kdims.insert(axis, KLONG)
    return tuple(dims), tuple(kdims)


@pytest.mark.parametrize("axis", [0, 1, 2], ids=["z", "y", "x"])
@pytest.mark.parametrize("n", LONG_AXES)
def test_long_axis_convolution(L, n, axis):
    """x runs k_rows_fwd / k_rows_inv, y the plain k_cols passes, z the merged k_cols pass with the K^ product"""
    if _emulated(L) and n in EMU_SKIPPED:
        pytest.skip("prime stage too long to emulate; runs on the GPU")
    dims, kdims = _long_axis_shape(axis, n)
    img, k = _random_conv(dims, kdims, seed=n + axis)
    exp = orc.inplace_cpu_convolution(img, k)
    got = img.copy()
    L.inplace_gpu_convolution(got, k)
    assert L.last_geometry() == NATIVE
    assert _strategy(L, dims) == (capi.STRATEGY_GENERIC, dims)
    if n in PRIMES:
        ref = _f64_convolution(img, k)
        print("prime %d on axis %s: vs oracle (max rel, rel L2) = (%.3g, %.3g); vs float64: library %.3g, oracle %.3g"
              % (n, "zyx"[axis], pc.max_rel(got, exp), pc.rel_l2(got, exp), pc.rel_l2(got, ref), pc.rel_l2(exp, ref)))
    _assert_conv_close(got, exp)


# ---- b. rejections ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("axis", [0, 1, 2], ids=["z", "y", "x"])
def test_axis_past_the_limit_is_rejected(L, axis):
    dims = [2, 3, 4]
    dims[axis] = MAX_AXIS + 1
    img = np.ones(dims, F32)
    before = img.copy()
    with pytest.raises(capi.LmvnError, match=LIMIT_MESSAGE):
        L.inplace_gpu_convolution(img, np.ones((1, 1, 1), F32))
    np.testing.assert_array_equal(img, before)  # output untouched on failure


_REJECT_SCRIPT = r"""
import faulthandler, sys, time
sys.path.insert(0, sys.argv[1])
from libmultiviewnative_b200 import capi
L = capi.Library(sys.argv[2])
for dims in [(1, 1, 12801), (1, 1, 2147483647), (2147483647, 1, 1), (1, 100000000, 1)]:
    # a watchdog thread ends the process if the call is still running after a second, even inside the library
    faulthandler.dump_traceback_later(1.0, exit=True)
    t0 = time.perf_counter()
    try:
        L.plan(dims, 1)
    except capi.LmvnError as e:
        faulthandler.cancel_dump_traceback_later()
        assert "exceeds the shared-memory transform limit" in str(e), e
        print("rejected", dims, "in %.4f s" % (time.perf_counter() - t0))
    else:
        raise SystemExit("not rejected: %s" % (dims,))
"""


def test_unbounded_extent_is_rejected_before_planning(E):
    """An axis of 10^8 or 2^31 - 1 points must be rejected by the shared-memory limit before the length is factorised
    or its twiddle table allocated (8 n bytes on host and device: 800 MB for 10^8 points, 16 GB for 2^31 - 1).  Each
    rejection must take less than a second, which only a check ahead of the twiddle table passes.  The calls run in a
    child process: a watchdog ends it when a call overruns, and the 60 s timeout catches a child that hangs anyway."""
    r = subprocess.run([sys.executable, "-c", _REJECT_SCRIPT, ROOT, E.path], capture_output=True, text=True,
                       timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("rejected") == 4, r.stdout


# ---- c. camera-frame deconvolution -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dims,lam", [((16, 2048, 2048), 0.006), ((16, 2160, 2560), 0.0)],
                         ids=["16x2048x2048", "16x2160x2560"])
def test_camera_frame_deconvolve(G, dims, lam):
    """one-shot call on sCMOS frames, 2 views, 15-point PSFs, against the pocketfft oracle after 1 and 3 iterations.
    The torch twin cannot serve at these shapes: with torch 2.11.0 (CPU, MKL), torch.fft.irfftn(torch.fft.rfftn(a),
    s=a.shape) of a float32 tensor of 16 x 1024 x 1024, 16 x 2048 x 2048 or even 16 x 2048 x 64 corrupts the heap
    ("malloc(): invalid size", abort with 1 thread, segmentation fault with 8), while 512 x 512 x 256 runs clean.  The
    forward transform alone is fine.  The oracle's loop carries nothing but psi, so 3 iterations are 1 iteration
    followed by 2 more."""
    d = make_views_fast(dims, 2, 15, 20240607)
    khats = ([orc.forwarded_kernel(k, dims, -1) for k in d["kernels1"]],
             [orc.forwarded_kernel(k, dims, -1) for k in d["kernels2"]])
    ck = {1: orc.inplace_cpu_deconvolve(d["psi0"], d["views"], None, None, d["weights"], 1, lam, 1e-4, nthreads=-1,
                                        khats=khats)}
    ck[3] = orc.inplace_cpu_deconvolve(ck[1], d["views"], None, None, d["weights"], 2, lam, 1e-4, nthreads=-1,
                                       khats=khats)
    res = {}
    for iters in (1, 3):
        psi = d["psi0"].copy()
        G.inplace_gpu_deconvolve(psi, d["views"], d["kernels1"], d["kernels2"], d["weights"], iters, lam, 1e-4)
        assert G.last_geometry() == NATIVE
        res[iters] = (pc.max_rel(psi, ck[iters]), pc.rel_l2(psi, ck[iters]))
    print("camera frame %s lam=%g: (max rel, rel L2) %s" % ("x".join(map(str, dims)), lam, res))
    assert _strategy(G, dims) == (capi.STRATEGY_GENERIC, dims)
    assert res[1][0] <= pc.PER_VOXEL_TOL_1_ITER, res
    assert res[1][1] <= pc.REL_L2_TOL_10_ITER and res[3][1] <= pc.REL_L2_TOL_10_ITER, res


def test_prime_axis_deconvolve(L):
    """reduced twin of the camera-frame case: a 1031-point prime x axis, 2 views, 1 and 2 iterations"""
    dims = (4, 8, 1031)
    d = make_views(dims, num_views=2, kernel_size=5, n_sources=12, workers=1)
    for iters in (1, 2):
        exp = orc.inplace_cpu_deconvolve(d["psi0"], d["views"], d["kernels1"], d["kernels2"], d["weights"], iters, 0.006,
                                         1e-4)
        psi = d["psi0"].copy()
        L.inplace_gpu_deconvolve(psi, d["views"], d["kernels1"], d["kernels2"], d["weights"], iters, 0.006, 1e-4)
        assert L.last_geometry() == NATIVE
        if iters == 1:
            assert pc.max_rel(psi, exp) <= pc.PER_VOXEL_TOL_1_ITER
        assert pc.rel_l2(psi, exp) <= pc.REL_L2_TOL_10_ITER
    assert _strategy(L, dims) == (capi.STRATEGY_GENERIC, dims)


# ---- d. zero-padded geometry through the generic passes -------------------------------------------------------------
def test_zero_padd_convolution_past_1024(L):
    """image x = 1000 with a 41-point kernel: padded to 1040, which create_padded cannot round to a fast extent"""
    dims, kdims = (4, 5, 1000), (3, 3, 41)
    img, k = _random_conv(dims, kdims, seed=21)
    padded, off = pc._zero_pad(img, kdims)
    exp = pc._crop(orc.inplace_cpu_convolution(padded, k), off, dims)
    L.set_padding(1)
    try:
        got = img.copy()
        L.inplace_gpu_convolution(got, k)
        assert L.last_geometry() == ZERO_PADDED
    finally:
        L.set_padding(0)
    assert _strategy(L, dims, kdims, "zero") == (capi.STRATEGY_GENERIC, (6, 7, 1040))
    _assert_conv_close(got, exp)


def test_zero_padd_deconvolve_past_1024(L):
    """41-point PSFs along a 1000-point x axis (the others clamp to 5 and 7): padded extents 10 x 14 x 1040"""
    dims = (6, 8, 1000)
    pc.case_zero_padd_deconvolve(L, dims, 41)
    assert L.last_geometry() == ZERO_PADDED
    assert _strategy(L, dims, (5, 7, 41), "zero") == (capi.STRATEGY_GENERIC, (10, 14, 1040))


# ---- e. the routing table ----------------------------------------------------------------------------------------------
def _fast_extent(n, x_axis):
    e = 64 if x_axis else 16
    while e <= 1024:
        if e >= n:
            return e
        e *= 2
    return 0


def _fused_shape_ok(nz, ny, nx):
    return (nx in (64, 128, 256, 512, 1024) and ny in (16, 32, 64, 128, 256, 512, 1024)
            and nz in (16, 32, 64, 128, 256, 512, 1024) and nz * ny % 128 == 0)


def _fast_extents(image, k):
    out = [_fast_extent(image[a] + k[a] - 1, a == 2) for a in range(3)]
    if min(out) <= 0:
        return None
    while out[0] * out[1] % 128 != 0 and out[1] < 1024:  # the rows kernels' 128-row granularity
        out[1] *= 2
    return tuple(out) if _fused_shape_ok(*out) else None


def expected_route(image, k, env):
    """csrc/api.cu restated: (geometry, strategy, plan extents) of a one-shot call with the AUTO strategy and circular
    padding.  Periodic embedding into fast-path extents >= image + k - 1 is taken when the fast path does not take the
    image itself, every kernel fits the image, and it costs at most LMVN_EMBED_MAX_BLOWUP (default 8) times the voxels."""
    native = (NATIVE, capi.STRATEGY_FUSED if _fused_shape_ok(*image) else capi.STRATEGY_GENERIC, tuple(image))
    if env.get("LMVN_EMBED", "1").startswith("0") or _fused_shape_ok(*image):
        return native
    if any(k[a] > image[a] for a in range(3)):
        return native
    fast = _fast_extents(image, k)
    if fast is None:
        return native
    blowup = float(np.prod(fast)) / float(np.prod(image))
    if blowup <= float(env.get("LMVN_EMBED_MAX_BLOWUP", 8.0)):
        return EMBEDDED, capi.STRATEGY_FUSED, fast
    return native


# (image zyx, kernel zyx, environment, expected geometry): the expectation is written out so that the table checks the
# restated rule too
ROUTES = [
    # image + k - 1 = 1023 / 1024 / 1025 along each axis
    ((6, 7, 1000), (3, 2, 24), {}, EMBEDDED),
    ((6, 7, 1000), (3, 2, 25), {}, EMBEDDED),
    ((6, 7, 1000), (3, 2, 26), {}, NATIVE),
    ((7, 1000, 20), (3, 24, 3), {}, EMBEDDED),
    ((7, 1000, 20), (3, 25, 3), {}, EMBEDDED),
    ((7, 1000, 20), (3, 26, 3), {}, NATIVE),
    ((1000, 7, 20), (24, 3, 3), {}, EMBEDDED),
    ((1000, 7, 20), (25, 3, 3), {}, EMBEDDED),
    ((1000, 7, 20), (26, 3, 3), {}, NATIVE),
    # the smallest fast extents: x = 63 / 64 / 65, y and z = 15 / 16 / 17
    ((16, 16, 63), (1, 1, 1), {}, EMBEDDED),
    ((16, 16, 64), (1, 1, 1), {}, NATIVE),  # the fast path natively
    ((16, 16, 65), (1, 1, 1), {}, EMBEDDED),
    ((16, 15, 64), (1, 1, 1), {}, EMBEDDED),
    ((16, 17, 64), (1, 1, 1), {}, EMBEDDED),
    ((15, 16, 64), (1, 1, 1), {}, EMBEDDED),
    ((17, 16, 64), (1, 1, 1), {}, EMBEDDED),
    ((16, 16, 64), (3, 3, 3), {}, NATIVE),  # taken natively however large the kernel: circular at the image extents
    ((14, 14, 62), (3, 3, 3), {}, EMBEDDED),  # image + k - 1 = 16 x 16 x 64 exactly
    ((14, 14, 63), (3, 3, 3), {}, EMBEDDED),  # x: 65 -> 128
    # blow-up just under, at and just over 8
    ((3, 12, 57), (1, 1, 1), {}, EMBEDDED),  # 7.98
    ((2, 16, 64), (1, 1, 1), {}, EMBEDDED),  # 8 exactly
    ((2, 16, 63), (1, 1, 1), {}, NATIVE),  # 8.13
    ((2, 16, 64), (1, 1, 1), {"LMVN_EMBED_MAX_BLOWUP": "7.99"}, NATIVE),
    ((1, 16, 64), (1, 1, 1), {"LMVN_EMBED_MAX_BLOWUP": "16"}, EMBEDDED),
    ((15, 16, 64), (1, 1, 1), {"LMVN_EMBED": "0"}, NATIVE),
    # plane counts nz * ny that are not multiples of 128 (5 x 9, 5 x 40)
    ((5, 9, 60), (3, 3, 3), {}, EMBEDDED),
    ((5, 40, 60), (1, 3, 5), {}, EMBEDDED),
    # thin stacks
    ((1, 16, 64), (1, 1, 1), {}, NATIVE),  # 16x the voxels
    ((2, 16, 64), (2, 1, 1), {}, EMBEDDED),
    ((3, 16, 64), (3, 1, 1), {}, EMBEDDED),
    ((3, 16, 64), (3, 3, 3), {}, NATIVE),  # 16 x 32 x 128: 21x the voxels
    # kernel extent equal to the image extent
    ((15, 16, 60), (15, 5, 5), {}, EMBEDDED),
    ((9, 10, 40), (9, 10, 40), {}, NATIVE),  # 36x the voxels
]


def _route_id(case):
    image, k, env, _ = case
    tag = "-".join("%s=%s" % kv for kv in env.items())
    return "x".join(map(str, image)) + "_k" + "x".join(map(str, k)) + ("_" + tag if tag else "")


@pytest.mark.parametrize("case", ROUTES, ids=[_route_id(c) for c in ROUTES])
def test_routing_table(E, case, monkeypatch):
    image, k, env, geometry = case
    for name in ("LMVN_EMBED", "LMVN_EMBED_MAX_BLOWUP"):
        monkeypatch.delenv(name, raising=False)
    for name, value in env.items():
        monkeypatch.setenv(name, value)
    route = expected_route(image, k, env)
    assert route[0] == geometry
    img, kern = _random_conv(image, k, seed=sum(image) + sum(k))
    got = img.copy()
    E.inplace_gpu_convolution(got, kern)
    assert E.last_geometry() == geometry
    if geometry == EMBEDDED:
        assert _strategy(E, image, k, "embedded") == route[1:]
        assert route[2][0] * route[2][1] % 128 == 0
    else:
        assert _strategy(E, image) == route[1:]
    _assert_conv_close(got, orc.inplace_cpu_convolution(img, kern))
