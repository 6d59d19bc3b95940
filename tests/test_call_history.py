"""A call's result must not depend on what ran before it in the process, or beside it.

State outlives a call in three places:
- destroyed handles park their device arena for the next handle on the device (csrc/engine.cu, take_parked / park),
  so every one-shot call after the first runs on memory full of an earlier call's psi, spectra and views;
- a persistent handle captures one sweep of the chained loop into a CUDA graph and replays it
  (Deconv::iterate); it must re-capture whenever lambda, min_value or the psi buffer changes;
- the block pipeline (blocks.run_pipelined) keeps two or three calls in flight per device.  They share the plan store,
  the FFT tables, the pinned staging ring and the thread-local error / geometry state.

Every result here is compared BIT FOR BIT with the same call made first thing in a fresh Python process.  That clean
result is anchored once per case to the oracle with the parity tolerances.  A fresh device allocation is zero on the
GPU and NaN in the emulator; a reused one holds plausible finite data, which hides under any tolerance.  So the tests
fill the parked arenas on purpose (lmvn_debug_fill_parked_arenas): with NaN, with zeros and with a finite pattern.

The emulator fixture runs the shared cases in the CPU suite; the `gpu` fixture runs them, the CUDA-graph sequences and
the concurrent calls on the product library.  Every run is a fixed list of calls, each made once.
"""
import json
import os
import subprocess
import sys
import threading
from functools import lru_cache

import numpy as np
import pytest

from libmultiviewnative_b200 import blocks, capi
from libmultiviewnative_b200.synthetic import make_views, make_views_fast
from oracle import mvn_oracle as orc
from tests import parity_cases as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
NATIVE, EMBEDDED, ZERO_PADDED = pc.GEOMETRY_NATIVE, pc.GEOMETRY_EMBEDDED, pc.GEOMETRY_ZERO_PADDED
FILLS = (0xFF, 0x00, 0x3F)  # NaN, zero, about 0.75 in every float
MIB = 1 << 20


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
def G():
    lib = capi.load()
    assert "sm_100a" in lib.version() and lib.num_devices() >= 1
    yield lib
    lib.release_cached_memory()


# ---- one call: a JSON spec and named arrays, so that a fresh process can make the same call ------------------------
def _deconv_call(dims, nviews, ksize, iters, lam=0.006, geometry=NATIVE, fast_data=False, seed=20240607, **extra):
    if fast_data:
        d = make_views_fast(dims, num_views=nviews, kernel_size=ksize, seed=seed)
    else:
        d = make_views(dims, num_views=nviews, kernel_size=ksize, n_sources=8, seed=seed, workers=1)
    arrays = {"psi": d["psi0"]}
    for v in range(nviews):
        arrays.update({f"view{v}": d["views"][v], f"weights{v}": d["weights"][v], f"k1_{v}": d["kernels1"][v],
                       f"k2_{v}": d["kernels2"][v]})
    spec = dict(kind="deconvolve", nviews=nviews, iters=iters, lam=lam, min_value=1e-4, geometry=geometry)
    spec.update(extra)
    return spec, arrays


def _conv_call(dims, kdims, geometry=NATIVE, **extra):
    rng = np.random.default_rng(41)
    k = rng.random(kdims, dtype=F32)
    spec = dict(kind="convolve", geometry=geometry)
    spec.update(extra)
    return spec, {"im": (rng.random(dims, dtype=F32) + 1).astype(F32), "kernel": (k / k.sum()).astype(F32)}


def _legacy_call(dims, ksize):
    d = make_views(dims, num_views=1, kernel_size=ksize, n_sources=4, workers=1)
    return dict(kind="iterate_fft_plain", geometry=NATIVE), {"inp": d["views"][0], "kernel": d["kernels1"][0]}


@lru_cache(maxsize=None)
def history_case(name):
    """(spec, arrays) of the calls every build runs on a dirty arena; `gpu_` cases only run on the B200."""
    if name == "native_split":  # fast path, Nyquist column as a compact plane behind the spectrum
        return _deconv_call((16, 16, 64), 2, 5, 2)
    if name == "native_whole_rows":  # Nyquist column inside the rows: pitch 33 -> 40, the pad columns are never written
        return _deconv_call((16, 16, 64), 2, 5, 2, env={"LMVN_SPLIT_NYQUIST": "0"})
    if name == "nx1024":  # wide rows, chained
        return _deconv_call((16, 16, 1024), 1, 3, 2)
    if name == "embedded":  # odd extents embedded periodically: psi / psi2 and the second spectrum buffer swap roles
        return _deconv_call((15, 15, 45), 2, 5, 3, geometry=EMBEDDED)
    if name == "zero_padd":  # k_place_box zero fill, zero_view_guard
        return _deconv_call((12, 12, 28), 2, 5, 2, geometry=ZERO_PADDED, padding=1)
    if name == "generic":
        return _deconv_call((9, 10, 15), 2, 5, 2, strategy=capi.STRATEGY_GENERIC)
    if name == "conv_native":
        return _conv_call((16, 16, 64), (5, 7, 3))
    if name == "conv_embedded":
        return _conv_call((20, 24, 50), (5, 7, 9), geometry=EMBEDDED)
    if name == "conv_zero_padd":
        return _conv_call((12, 12, 28), (5, 5, 5), geometry=ZERO_PADDED, padding=1)
    if name == "legacy_plain":
        return _legacy_call((8, 8, 16), 5)
    if name == "gpu_config4_block":  # BASELINE config 4: 256^3 blocks, 41^3 PSFs
        return _deconv_call((256, 256, 256), 2, 41, 3, fast_data=True)
    raise KeyError(name)


SHARED_CASES = ["native_split", "native_whole_rows", "nx1024", "embedded", "zero_padd", "generic", "conv_native",
                "conv_embedded", "conv_zero_padd", "legacy_plain"]


class _Settings:
    """the process-wide padding mode and strategy of a spec, restored to the defaults afterwards"""

    def __init__(self, L, spec):
        self.L, self.spec = L, spec

    def __enter__(self):
        self.L.set_padding(self.spec.get("padding", 0))
        self.L.set_default_strategy(self.spec.get("strategy", capi.STRATEGY_AUTO))

    def __exit__(self, *exc):
        self.L.set_padding(0)
        self.L.set_default_strategy(capi.STRATEGY_AUTO)


def _views(spec, a):
    n = spec["nviews"]
    return ([a[f"view{v}"] for v in range(n)], [a[f"k1_{v}"] for v in range(n)], [a[f"k2_{v}"] for v in range(n)],
            [a[f"weights{v}"] for v in range(n)])


def run_call(L, spec, a):
    """Makes the call; returns (result, lmvn_last_geometry of this thread)."""
    with _Settings(L, spec):
        if spec["kind"] == "deconvolve":
            out = a["psi"].copy()
            views, k1, k2, w = _views(spec, a)
            L.inplace_gpu_deconvolve(out, views, k1, k2, w, spec["iters"], spec["lam"], spec["min_value"])
        elif spec["kind"] == "convolve":
            out = a["im"].copy()
            L.inplace_gpu_convolution(out, a["kernel"])
        else:
            out = L.iterate_fft_plain(a["inp"], a["kernel"])
        return out, L.last_geometry()


_CLEAN_PROCESS = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from libmultiviewnative_b200.capi import Library
from tests.test_call_history import run_call
with open(sys.argv[3]) as f:
    spec = json.load(f)
with np.load(sys.argv[4]) as z:
    arrays = {k: z[k] for k in z.files}
out, geometry = run_call(Library(sys.argv[2]), spec, arrays)
np.save(sys.argv[5], out)
print(geometry)
"""


def clean_process_result(L, spec, arrays, tmp_path):
    """The same call as the first and only call of a fresh interpreter, on the same library file."""
    spec_path, npz, out = (str(tmp_path / n) for n in ("call.json", "call.npz", "clean.npy"))
    with open(spec_path, "w") as f:
        json.dump(spec, f)
    np.savez(npz, **arrays)
    env = dict(os.environ)
    env.update(spec.get("env", {}))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _CLEAN_PROCESS, ROOT, L.path,
                                                                           spec_path, npz, out]
    res = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    if spec["kind"] != "iterate_fft_plain":  # the legacy entry points do not report a geometry
        assert int(res.stdout.split()[-1]) == spec["geometry"]
    return np.load(out)


def _zero_padded(a, kmax):
    return pc._zero_pad(np.asarray(a, dtype=F32), kmax)


def anchor_to_oracle(spec, a, got):
    """The clean result against the oracle, with the parity suite's tolerances."""
    if spec["kind"] == "deconvolve":
        views, k1, k2, w = _views(spec, a)
        iters, lam, mv = spec["iters"], spec["lam"], spec["min_value"]
        if spec.get("padding"):
            kmax = [max(k.shape[ax] for k in k1 + k2) for ax in range(3)]
            ppsi, off = _zero_padded(a["psi"], kmax)
            exp = pc._crop(orc.inplace_cpu_deconvolve(ppsi, [_zero_padded(v, kmax)[0] for v in views], k1, k2,
                                                      [_zero_padded(x, kmax)[0] for x in w], iters, lam, mv,
                                                      nthreads=-1, zero_view_guard=True), off, a["psi"].shape)
        elif a["psi"].size > (1 << 20):
            exp = orc.inplace_cpu_deconvolve_torch(a["psi"], views, k1, k2, w, iters, lam, mv)
        else:
            exp = orc.inplace_cpu_deconvolve(a["psi"], views, k1, k2, w, iters, lam, mv, nthreads=-1)
        if iters <= 2:
            assert pc.max_rel(got, exp) <= pc.PER_VOXEL_TOL_1_ITER
        assert pc.rel_l2(got, exp) <= pc.REL_L2_TOL_10_ITER
    elif spec["kind"] == "convolve":
        im, k = a["im"], a["kernel"]
        if spec.get("padding"):
            padded, off = _zero_padded(im, k.shape)
            exp = pc._crop(orc.inplace_cpu_convolution(padded, k), off, im.shape)
        else:
            exp = orc.inplace_cpu_convolution(im, k)
        assert pc.rel_l2(got, exp) <= 1e-5
        assert pc.max_rel(got, exp) <= pc.PER_VOXEL_TOL_1_ITER
    else:
        inp, k1 = a["inp"], a["kernel"]
        exp = orc.inplace_cpu_deconvolve(inp, [inp], [k1], [np.full(k1.shape, 0.1, F32)], [np.ones_like(inp)], 1, 0.0,
                                         1e-4)
        assert pc.max_rel(got, exp) <= pc.PER_VOXEL_TOL_1_ITER


def _plan_like(L, spec, a):
    """A persistent handle of the geometry the one-shot call uses."""
    if spec["kind"] == "deconvolve":
        shape, nviews = a["psi"].shape, spec["nviews"]
        _, k1, k2, _ = _views(spec, a)
        kmax = [max(k.shape[ax] for k in k1 + k2) for ax in range(3)]
    else:
        shape, nviews = (a["im"] if "im" in a else a["inp"]).shape, 1
        kmax = list(a["kernel"].shape)
    geometry = {NATIVE: "native", EMBEDDED: "embedded", ZERO_PADDED: "zero"}[spec["geometry"]]
    with _Settings(L, spec):
        return L.plan(shape, nviews, -1, max_kernel_dims=None if geometry == "native" else kmax,
                      geometry=geometry)


def _target_arena(L, spec, a):
    """(arena bytes, working extents) of the handle the one-shot call creates"""
    with _plan_like(L, spec, a) as p:
        info = p.info()
        out = int(info.arena_bytes), tuple(info.dims)
    L.release_cached_memory()
    return out


def _park_donor(L, spec, a):
    """Parks the arena of a handle of another shape that the target's request takes: larger than the target needs
    (its buffers sit at other offsets than the arena's last owner's) and inside the best-fit window of take_parked
    (at most 1.5 x the request + 64 MiB).  Returns the donor's dims, its bytes and the target's."""
    need, (z, y, x) = _target_arena(L, spec, a)
    nviews = spec.get("nviews", 1)
    with _Settings(L, spec):
        for dims in ((z, y, x + 8), (z, y, x + 24), (z + 2, y, x), (z, y, x + x // 2), (z, y, 2 * x)):
            with L.plan(dims, nviews) as p:
                got = int(p.info().arena_bytes)
            if need < got <= need + need // 2 + 64 * MIB:
                L.release_cached_memory()
                L.plan(dims, nviews).close()
                return dims, got, need
            L.release_cached_memory()
    raise AssertionError(f"no donor arena inside the best-fit window of {need} bytes")


def check_dirty_arenas(L, name, tmp_path, monkeypatch):
    spec, a = history_case(name)
    for k, v in spec.get("env", {}).items():
        monkeypatch.setenv(k, v)
    clean = clean_process_result(L, spec, a, tmp_path)
    anchor_to_oracle(spec, a, clean)

    L.release_cached_memory()
    got, geometry = run_call(L, spec, a)  # parks its arena
    if spec["kind"] != "iterate_fft_plain":
        assert geometry == spec["geometry"]
    np.testing.assert_array_equal(got, clean, err_msg="after other calls in this process")
    for byte in FILLS:
        L.fill_parked_arenas(byte)
        got, _ = run_call(L, spec, a)
        np.testing.assert_array_equal(got, clean, err_msg=f"own arena filled with {byte:#04x}")

    L.release_cached_memory()
    dims, donor, need = _park_donor(L, spec, a)
    assert need < donor <= need + need // 2 + 64 * MIB
    for byte in (0xFF, 0x3F):
        L.fill_parked_arenas(byte)
        got, _ = run_call(L, spec, a)
        np.testing.assert_array_equal(got, clean, err_msg=f"arena of a {dims} handle filled with {byte:#04x}")
    L.release_cached_memory()


# ---- 1. dirty arenas ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SHARED_CASES)
def test_dirty_arena_gives_the_clean_process_result(L, name, tmp_path, monkeypatch):
    check_dirty_arenas(L, name, tmp_path, monkeypatch)


@pytest.mark.gpu
def test_dirty_arena_config4_block(G, tmp_path, monkeypatch):
    check_dirty_arenas(G, "gpu_config4_block", tmp_path, monkeypatch)


def test_fill_parked_arenas_without_arenas_is_a_no_op(L):
    L.release_cached_memory()
    L.fill_parked_arenas(0xFF)


# ---- 2. a rejected call leaves no trace ----------------------------------------------------------------------------------
def test_rejected_call_leaves_no_trace(L):
    """the second call fails after view 0 was uploaded (view 1's kernel is larger than the image): psi stays as it
    was, and the next good call gives the bits of the first"""
    dims = (16, 16, 64) if "emu" in L.version().lower() else (64, 128, 256)  # GPU: 8 MiB views go through the staging ring
    spec, a = _deconv_call(dims, 2, 5, 3)
    first, _ = run_call(L, spec, a)
    views, k1, k2, w = _views(spec, a)
    psi = a["psi"].copy()
    with pytest.raises(capi.LmvnError, match="does not fit"):
        L.inplace_gpu_deconvolve(psi, views, [k1[0], np.ones((dims[0] + 1, 3, 3), F32)], k2, w, 3, 0.006, 1e-4)
    np.testing.assert_array_equal(psi, a["psi"])
    again, _ = run_call(L, spec, a)
    np.testing.assert_array_equal(again, first)


# ---- 3. CUDA-graph replay of the sweep (the emulator has no graphs) ---------------------------------------------------------
def _graph_sequence(p, new_psi):
    """psi after each step; each of steps 2-5 changes ONE thing the captured sweep depends on, or nothing"""
    snaps = []
    p.iterate(4, 0.006)
    snaps.append(p.get_psi())
    p.iterate(4, 0.0)  # lambda changed
    snaps.append(p.get_psi())
    p.iterate(4, 0.0, min_value=1e-2)  # min_value changed
    snaps.append(p.get_psi())
    p.convolve(0, 1)  # swaps psi and integral: only the psi buffer differs from the last capture
    p.iterate(3, 0.0, min_value=1e-2)
    snaps.append(p.get_psi())
    p.convolve(0, 1)
    p.convolve(0, 1)  # psi is back at the buffer of the last capture: replayed as captured
    p.iterate(3, 0.0, min_value=1e-2)
    snaps.append(p.get_psi())
    p.set_psi(new_psi)
    p.iterate(5, 0.006)
    snaps.append(p.get_psi())
    return snaps


def _loaded_plan(G, d):
    p = G.plan(d["psi0"].shape, len(d["views"]))
    for v in range(len(d["views"])):
        p.set_view(v, d["views"][v], d["weights"][v], d["kernels1"][v], d["kernels2"][v])
    p.set_psi(d["psi0"])
    return p


@lru_cache(maxsize=None)
def _graph_data(dims):
    return make_views_fast(dims, num_views=1 if dims == (512, 512, 256) else 2, kernel_size=21, seed=7)


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(128, 128, 128), (64, 64, 1024), (512, 512, 256)], ids=lambda d: "x".join(map(str, d)))
def test_graph_replay_equals_plain_launches(G, dims, monkeypatch):
    d = _graph_data(dims)
    new_psi = (d["views"][-1] * F32(0.9) + F32(1.0)).astype(F32)
    runs = {}
    for graph in ("1", "0"):
        monkeypatch.setenv("LMVN_GRAPH", graph)  # read when the plan is created
        with _loaded_plan(G, d) as p:
            runs[graph] = _graph_sequence(p, new_psi)
    for step, (a, b) in enumerate(zip(runs["1"], runs["0"]), 1):
        np.testing.assert_array_equal(a, b, err_msg=f"graph step {step}")
    assert not np.array_equal(runs["1"][0], runs["1"][1])  # the steps do change psi

    exp = orc.inplace_cpu_deconvolve_torch(new_psi, d["views"], d["kernels1"], d["kernels2"], d["weights"], 5, 0.006, 1e-4)
    assert pc.rel_l2(runs["1"][-1], exp) <= pc.REL_L2_TOL_10_ITER
    monkeypatch.setenv("LMVN_GRAPH", "1")
    with _loaded_plan(G, d) as p:
        p.iterate(1, 0.006)
        one = p.get_psi()
    exp = orc.inplace_cpu_deconvolve_torch(d["psi0"], d["views"], d["kernels1"], d["kernels2"], d["weights"], 1, 0.006, 1e-4)
    assert pc.max_rel(one, exp) <= pc.PER_VOXEL_TOL_1_ITER


# ---- 4. calls side by side ------------------------------------------------------------------------------------------------
PIPELINE_SHAPES = [(256, 256, 256), (200, 256, 256), (101, 105, 225)]  # native; 52 MB = four staging chunks; embedded


@lru_cache(maxsize=None)
def _pipeline_base(i):
    return make_views_fast(PIPELINE_SHAPES[i], num_views=2, kernel_size=21, seed=11 + i)


def _pinned(a):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy()  # shares the pinned storage; the tensor is kept alive by the array's base


def _pipeline_block(b):
    """block b: shape b mod 3, data scaled per block; odd blocks hand the library page-locked stacks"""
    base, s = _pipeline_base(b % 3), F32(1.0 + 0.25 * (b // 3))
    conv = _pinned if b % 2 else np.ascontiguousarray
    return dict(psi0=conv(base["psi0"] * s), views=[conv(v * s) for v in base["views"]], weights=[conv(w) for w in base["weights"]],
                kernels1=base["kernels1"], kernels2=base["kernels2"])


@pytest.mark.gpu
@pytest.mark.parametrize("depth,iters", [(2, 3), (3, 5)])
def test_block_pipeline_equals_blocks_run_alone(G, depth, iters):
    """two calls in flight (depth 3: three, with two park slots one arena is allocated fresh); the graph capture of
    one call overlaps the uploads and launches of the other"""
    G.release_cached_memory()
    got = blocks.run_pipelined(G, _pipeline_block, range(6), iters, 0.006, 1e-4, device=0, depth=depth)
    assert sorted(got) == list(range(6))
    for b in range(6):
        alone = blocks.deconvolve_block(G, _pipeline_block(b), iters, 0.006, 1e-4, 0)
        np.testing.assert_array_equal(got[b], alone, err_msg=f"block {b} ({PIPELINE_SHAPES[b % 3]})")
    assert G.last_geometry() == EMBEDDED  # block 5
    d = _pipeline_block(5)
    exp = orc.inplace_cpu_deconvolve_torch(d["psi0"], d["views"], d["kernels1"], d["kernels2"], d["weights"], iters, 0.006,
                                           1e-4)
    assert pc.rel_l2(got[5], exp) <= pc.REL_L2_TOL_10_ITER


def _plan_steps(G, d, p_box):
    """a persistent handle's calls, one per step; get_psi steps yield a snapshot"""
    def create():
        p_box.append(G.plan(d["psi0"].shape, 2))

    steps = [create]
    for v in range(2):
        steps.append(lambda v=v: p_box[0].set_view(v, d["views"][v], d["weights"][v], d["kernels1"][v], d["kernels2"][v]))
    steps += [lambda: p_box[0].set_psi(d["psi0"]), lambda: p_box[0].iterate(4, 0.006), lambda: p_box[0].get_psi(),
              lambda: p_box[0].iterate(3, 0.0), lambda: p_box[0].get_psi(), lambda: p_box[0].iterate(1, 0.006),
              lambda: p_box[0].get_psi(), lambda: p_box[0].close()]
    return steps


def _snapshots(results):
    return [r for r in results if isinstance(r, np.ndarray)]


@pytest.mark.gpu
@pytest.mark.parametrize("dims_b", [(128, 128, 128), (64, 128, 256)], ids=["same_dims", "other_dims"])
def test_two_plans_interleaved_on_one_thread(G, dims_b):
    da = make_views_fast((128, 128, 128), num_views=2, kernel_size=21, seed=3)
    db = make_views_fast(dims_b, num_views=2, kernel_size=21, seed=4)
    solo = {}
    for key, d in (("a", da), ("b", db)):
        solo[key] = _snapshots([s() for s in _plan_steps(G, d, [])])
    box_a, box_b = [], []
    sa, sb = _plan_steps(G, da, box_a), _plan_steps(G, db, box_b)
    ra, rb = [], []
    for step_a, step_b in zip(sa, sb):
        ra.append(step_a())
        rb.append(step_b())
    for key, got in (("a", _snapshots(ra)), ("b", _snapshots(rb))):
        assert len(got) == len(solo[key]) == 3
        for i, (x, y) in enumerate(zip(got, solo[key])):
            np.testing.assert_array_equal(x, y, err_msg=f"plan {key}, snapshot {i}")


@pytest.mark.gpu
def test_error_and_geometry_are_per_thread(G):
    """while one thread runs a good embedded call, another makes a call that is rejected after its plan was made"""
    d = _pipeline_base(2)
    solo = blocks.deconvolve_block(G, d, 5, 0.006, 1e-4, 0)
    bad = make_views_fast((64, 64, 64), num_views=2, kernel_size=5, seed=5)
    start = threading.Barrier(2)
    out, errors = {}, []

    def good():
        try:
            start.wait()
            out["psi"] = blocks.deconvolve_block(G, d, 5, 0.006, 1e-4, 0)
            out["geometry"] = G.last_geometry()
        except BaseException as exc:
            errors.append(exc)

    def rejected():
        try:
            start.wait()
            psi = bad["psi0"].copy()
            with pytest.raises(capi.LmvnError) as info:
                G.inplace_gpu_deconvolve(psi, bad["views"], [bad["kernels1"][0], np.ones((65, 3, 3), F32)],
                                         bad["kernels2"], bad["weights"], 2, 0.006, 1e-4)
            out["error"] = str(info.value)
            out["bad_geometry"] = G.last_geometry()
        except BaseException as exc:
            errors.append(exc)

    threads = [threading.Thread(target=good), threading.Thread(target=rejected)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    assert out["geometry"] == EMBEDDED and out["bad_geometry"] == NATIVE
    assert "extent 65 along axis 0 does not fit the image extent 64" in out["error"]
    np.testing.assert_array_equal(out["psi"], solo)


@pytest.mark.gpu
def test_two_gpus_equal_device_0(G):
    if G.num_devices() < 2:
        pytest.skip("needs two GPUs")
    blks = [dict(make_views_fast((128, 128, 128), num_views=2, kernel_size=21, seed=20 + b)) for b in range(4)]
    got = blocks.run_threads(G, blks, [0, 1], 3, 0.006, 1e-4)
    for b in range(4):
        np.testing.assert_array_equal(got[b], blocks.deconvolve_block(G, blks[b], 3, 0.006, 1e-4, 0), err_msg=f"block {b}")
