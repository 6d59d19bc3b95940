"""ctypes binding of libmultiviewnative.so -- the host-side mirror of the
reference interface (ref: inc/multiviewnative.h) for Python callers.

The wrappers keep the reference's names, argument meaning and in-place
semantics (``psi`` / ``im`` are numpy float32 arrays updated in place; dims are
taken from the array shapes as {z, y, x}).  Unlike the void C functions they
raise ``LmvnError`` when the library reports a failure, so nothing can pass
silently.  There is no CPU fallback: if the CUDA library has not been built,
loading raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIBRARY = os.path.join(_PKG, "lib", "libmultiviewnative.so")

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)


class ViewData(C.Structure):
    """struct view_data (ref: inc/multiviewnative.h:15-26), 64 bytes."""
    _fields_ = [
        ("image_", c_float_p), ("kernel1_", c_float_p), ("kernel2_", c_float_p), ("weights_", c_float_p),
        ("image_dims_", c_int_p), ("kernel1_dims_", c_int_p), ("kernel2_dims_", c_int_p), ("weights_dims_", c_int_p),
    ]


class Workspace(C.Structure):
    """struct workspace (ref: inc/multiviewnative.h:28-35), 32 bytes, passed by value."""
    _fields_ = [
        ("data_", C.POINTER(ViewData)), ("num_views_", C.c_ushort), ("lambda_", C.c_double),
        ("minValue_", C.c_float), ("num_iterations_", C.c_int),
    ]


class PlanInfo(C.Structure):
    _fields_ = [
        ("dims", C.c_int * 3), ("num_views", C.c_int), ("device", C.c_int), ("strategy", C.c_int),
        ("launches_per_view_iteration", C.c_int), ("arena_bytes", C.c_ulonglong), ("real_bytes", C.c_ulonglong),
        ("spectrum_bytes", C.c_ulonglong), ("alg_bytes_per_view_iteration", C.c_ulonglong),
    ]


class DistInfo(C.Structure):
    """struct lmvn_dist_info (include/lmvn_b200.h)."""
    _fields_ = [
        ("dims", C.c_int * 3), ("num_views", C.c_int), ("rank", C.c_int), ("world", C.c_int), ("device", C.c_int),
        ("planes_per_rank", C.c_int), ("rows_per_rank", C.c_int), ("spectrum_pitch", C.c_int),
        ("arena_bytes", C.c_ulonglong), ("exchange_bytes", C.c_ulonglong),
        ("alg_bytes_per_view_iteration", C.c_ulonglong), ("exchange_bytes_per_view_iteration", C.c_ulonglong),
    ]


assert C.sizeof(ViewData) == 64 and C.sizeof(Workspace) == 32

# every symbol include/multiviewnative.h and include/lmvn_b200.h declare
REFERENCE_SYMBOLS = [
    "inplace_cpu_convolution", "inplace_cpu_deconvolve", "inplace_gpu_convolution", "inplace_gpu_deconvolve",
    "convolution3DfftCUDAInPlace", "convolution3DfftCUDAInPlace_core", "compute_quotient", "compute_final_values",
    "iterate_fft_plain", "iterate_fft_tikhonov", "selectDeviceWithHighestComputeCapability",
    "getCUDAcomputeCapabilityMinorVersion", "getCUDAcomputeCapabilityMajorVersion", "getNumDevicesCUDA",
    "getNameDeviceCUDA", "getMemDeviceCUDA",
]
EXTENSION_SYMBOLS = [
    "lmvn_last_error", "lmvn_clear_error", "lmvn_version", "lmvn_set_default_strategy", "lmvn_release_cached_memory",
    "lmvn_plan_create", "lmvn_set_padding", "lmvn_plan_create_zero_padded", "lmvn_plan_create_embedded",
    "lmvn_last_geometry",
    "lmvn_plan_destroy", "lmvn_plan_get_info", "lmvn_plan_set_view", "lmvn_plan_set_psi", "lmvn_plan_get_psi",
    "lmvn_plan_iterate", "lmvn_plan_convolve", "lmvn_plan_profile", "lmvn_plan_synchronize", "lmvn_debug_rfftn", "lmvn_debug_irfftn",
    "lmvn_debug_fill_parked_arenas",
    "lmvn_dist_create", "lmvn_dist_destroy", "lmvn_dist_get_info", "lmvn_dist_export_handle", "lmvn_dist_connect_ipc",
    "lmvn_dist_connect_local", "lmvn_dist_set_view_slab", "lmvn_dist_set_psi_slab", "lmvn_dist_get_psi_slab",
    "lmvn_dist_psf_phase", "lmvn_dist_conv_phase", "lmvn_dist_barrier", "lmvn_dist_reset_barrier", "lmvn_dist_iterate",
    "lmvn_dist_synchronize",
    "lmvn_dist_set_stream", "lmvn_dist_set_staged", "lmvn_dist_buffer",
]

STRATEGY_AUTO, STRATEGY_GENERIC, STRATEGY_FUSED = 0, 1, 2


class LmvnError(RuntimeError):
    pass


def _f32(a, name="array") -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.float32 or not a.flags["C_CONTIGUOUS"]:
        raise TypeError(f"{name} must be a C-contiguous float32 array")
    return a


def _fp(a: np.ndarray):
    return a.ctypes.data_as(c_float_p)


def _dims(shape) -> "C.Array":
    if len(shape) != 3:
        raise ValueError("stacks must be 3-D {z, y, x}")
    return (C.c_int * 3)(*[int(s) for s in shape])


class Library:
    """A loaded libmultiviewnative.so."""

    def __init__(self, path: Optional[str] = None):
        path = path or os.environ.get("LMVN_LIBRARY") or DEFAULT_LIBRARY
        if not os.path.exists(path):
            raise LmvnError(
                f"{path} not found: the CUDA library has not been built "
                "(python -m libmultiviewnative_b200._build cuda); there is no CPU fallback")
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        L.lmvn_version.restype = C.c_char_p
        # the host-emulator test build (tests/emu) runs one kernel at a time on fibers: not re-entrant
        self.reentrant = b"emu" not in (L.lmvn_version() or b"").lower()
        L.lmvn_last_error.restype = C.c_char_p
        L.lmvn_version.restype = C.c_char_p
        L.lmvn_clear_error.restype = None
        L.lmvn_release_cached_memory.restype = None
        L.inplace_gpu_deconvolve.argtypes = [c_float_p, Workspace, C.c_int]
        L.inplace_gpu_deconvolve.restype = None
        L.inplace_cpu_deconvolve.argtypes = [c_float_p, Workspace, C.c_int]
        L.inplace_cpu_deconvolve.restype = None
        for fn in (L.inplace_gpu_convolution, L.inplace_cpu_convolution, L.convolution3DfftCUDAInPlace):
            fn.argtypes = [c_float_p, c_int_p, c_float_p, c_int_p, C.c_int]
            fn.restype = None
        L.compute_quotient.argtypes = [c_float_p, c_float_p, C.c_size_t, C.c_int]
        L.compute_quotient.restype = None
        L.compute_final_values.argtypes = [c_float_p, c_float_p, c_float_p, C.c_size_t, C.c_float, C.c_double, C.c_int]
        L.compute_final_values.restype = None
        L.iterate_fft_plain.argtypes = [c_float_p, c_float_p, c_float_p, c_int_p, c_int_p, C.c_int]
        L.iterate_fft_plain.restype = None
        L.iterate_fft_tikhonov.argtypes = [c_float_p, c_float_p, c_float_p, c_int_p, c_int_p, C.c_size_t, C.c_float,
                                           C.c_double, C.c_int]
        L.iterate_fft_tikhonov.restype = None
        L.getNameDeviceCUDA.argtypes = [C.c_int, C.c_char_p]
        L.getNameDeviceCUDA.restype = None
        L.getMemDeviceCUDA.restype = C.c_longlong
        L.lmvn_plan_create.argtypes = [C.POINTER(C.c_void_p), c_int_p, C.c_int, C.c_int]
        L.lmvn_plan_create_zero_padded.argtypes = [C.POINTER(C.c_void_p), c_int_p, c_int_p, C.c_int, C.c_int]
        L.lmvn_plan_create_embedded.argtypes = [C.POINTER(C.c_void_p), c_int_p, c_int_p, C.c_int, C.c_int]
        L.lmvn_plan_destroy.argtypes = [C.c_void_p]
        L.lmvn_plan_destroy.restype = None
        L.lmvn_plan_get_info.argtypes = [C.c_void_p, C.POINTER(PlanInfo)]
        L.lmvn_plan_set_view.argtypes = [C.c_void_p, C.c_int, c_float_p, c_float_p, c_float_p, c_int_p, c_float_p, c_int_p]
        L.lmvn_plan_set_psi.argtypes = [C.c_void_p, c_float_p]
        L.lmvn_plan_get_psi.argtypes = [C.c_void_p, c_float_p]
        L.lmvn_plan_iterate.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_float, c_float_p]
        L.lmvn_plan_convolve.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_float_p]
        L.lmvn_plan_synchronize.argtypes = [C.c_void_p]
        L.lmvn_plan_profile.argtypes = [C.c_void_p, C.c_double, C.c_float, C.c_int, C.c_char_p, c_float_p,
                                        C.POINTER(C.c_ulonglong), c_int_p]
        L.lmvn_dist_create.argtypes = [C.POINTER(C.c_void_p), c_int_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.lmvn_dist_destroy.argtypes = [C.c_void_p]
        L.lmvn_dist_destroy.restype = None
        L.lmvn_dist_get_info.argtypes = [C.c_void_p, C.POINTER(DistInfo)]
        L.lmvn_dist_export_handle.argtypes = [C.c_void_p, C.c_char_p]
        L.lmvn_dist_connect_ipc.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
        L.lmvn_dist_connect_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.lmvn_dist_set_view_slab.argtypes = [C.c_void_p, C.c_int, c_float_p, c_float_p]
        L.lmvn_dist_set_psi_slab.argtypes = [C.c_void_p, c_float_p]
        L.lmvn_dist_get_psi_slab.argtypes = [C.c_void_p, c_float_p]
        L.lmvn_dist_psf_phase.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_float_p, c_int_p]
        L.lmvn_dist_conv_phase.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_float]
        L.lmvn_dist_barrier.argtypes = [C.c_void_p]
        L.lmvn_dist_reset_barrier.argtypes = [C.c_void_p]
        L.lmvn_dist_iterate.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_float, c_float_p]
        L.lmvn_dist_synchronize.argtypes = [C.c_void_p]
        L.lmvn_dist_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.lmvn_dist_set_staged.argtypes = [C.c_void_p, C.c_int]
        L.lmvn_dist_buffer.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_ulonglong)]
        L.lmvn_debug_rfftn.argtypes = [c_float_p, c_int_p, c_float_p, C.c_int]
        L.lmvn_debug_irfftn.argtypes = [c_float_p, c_int_p, c_float_p, C.c_int]
        L.lmvn_debug_fill_parked_arenas.argtypes = [C.c_int]

    def set_padding(self, mode: int):
        """0: circular at the image extents (the CPU path, default); 1: zero_padd (the reference's GPU geometry)."""
        self._check(self.lib.lmvn_set_padding(int(mode)), "lmvn_set_padding")

    def last_geometry(self) -> int:
        """1: native extents, 2: periodic embedding into power-of-two extents, 3: zero padded (last one-shot call)."""
        return int(self.lib.lmvn_last_geometry())

    def release_cached_memory(self):
        self.lib.lmvn_release_cached_memory()

    def fill_parked_arenas(self, byte: int):
        """Sets every byte of the arenas parked for later calls to `byte` (tests: the next call runs on dirty memory)."""
        self._check(self.lib.lmvn_debug_fill_parked_arenas(int(byte)), "lmvn_debug_fill_parked_arenas")

    # -- error plumbing ----------------------------------------------------
    def last_error(self) -> str:
        return (self.lib.lmvn_last_error() or b"").decode()

    def _check_void(self, what: str):
        err = self.last_error()
        if err:
            self.lib.lmvn_clear_error()
            raise LmvnError(f"{what}: {err}")

    def _check(self, rc: int, what: str):
        if rc != 0:
            err = self.last_error()
            self.lib.lmvn_clear_error()
            raise LmvnError(f"{what}: {err}")

    def version(self) -> str:
        return self.lib.lmvn_version().decode()

    def set_default_strategy(self, strategy: int):
        self._check(self.lib.lmvn_set_default_strategy(int(strategy)), "lmvn_set_default_strategy")

    # -- reference API -------------------------------------------------------
    def _workspace(self, views, kernels1, kernels2, weights, num_iterations, lam, min_value):
        n = len(views)
        if not (len(kernels1) == len(kernels2) == len(weights) == n):
            raise ValueError("views, kernels and weights must have the same length")
        keep = []
        arr = (ViewData * n)()
        for v in range(n):
            im, k1, k2, w = (_f32(views[v], "view"), _f32(kernels1[v], "kernel1"), _f32(kernels2[v], "kernel2"),
                             _f32(weights[v], "weights"))
            d_im, d_k1, d_k2, d_w = _dims(im.shape), _dims(k1.shape), _dims(k2.shape), _dims(w.shape)
            keep += [im, k1, k2, w, d_im, d_k1, d_k2, d_w]
            arr[v].image_, arr[v].kernel1_, arr[v].kernel2_, arr[v].weights_ = _fp(im), _fp(k1), _fp(k2), _fp(w)
            arr[v].image_dims_ = C.cast(d_im, c_int_p)
            arr[v].kernel1_dims_ = C.cast(d_k1, c_int_p)
            arr[v].kernel2_dims_ = C.cast(d_k2, c_int_p)
            arr[v].weights_dims_ = C.cast(d_w, c_int_p)
        ws = Workspace()
        ws.data_ = C.cast(arr, C.POINTER(ViewData))
        ws.num_views_ = n
        ws.lambda_ = float(lam)
        ws.minValue_ = float(min_value)
        ws.num_iterations_ = int(num_iterations)
        keep.append(arr)
        return ws, keep

    def inplace_gpu_deconvolve(self, psi, views, kernels1, kernels2, weights, num_iterations, lam=0.0,
                               min_value=1e-4, device=-1):
        """ref: inc/multiviewnative.h:66 -- psi (float32, shape of view 0) is updated in place."""
        psi = _f32(psi, "psi")
        ws, keep = self._workspace(views, kernels1, kernels2, weights, num_iterations, lam, min_value)
        self.lib.lmvn_clear_error()
        self.lib.inplace_gpu_deconvolve(_fp(psi), ws, int(device))
        self._check_void("inplace_gpu_deconvolve")
        del keep
        return psi

    def inplace_cpu_deconvolve(self, psi, views, kernels1, kernels2, weights, num_iterations, lam=0.0,
                               min_value=1e-4, nthreads=1):
        psi = _f32(psi, "psi")
        ws, keep = self._workspace(views, kernels1, kernels2, weights, num_iterations, lam, min_value)
        self.lib.inplace_cpu_deconvolve(_fp(psi), ws, int(nthreads))
        del keep
        return psi

    def _conv(self, fn, name, im, kernel, last):
        im, kernel = _f32(im, "im"), _f32(kernel, "kernel")
        self.lib.lmvn_clear_error()
        fn(_fp(im), C.cast(_dims(im.shape), c_int_p), _fp(kernel), C.cast(_dims(kernel.shape), c_int_p), int(last))
        self._check_void(name)
        return im

    def inplace_gpu_convolution(self, im, kernel, device=-1):
        """ref: inc/multiviewnative.h:59 -- circular convolution at im's extents, in place."""
        return self._conv(self.lib.inplace_gpu_convolution, "inplace_gpu_convolution", im, kernel, device)

    def inplace_cpu_convolution(self, im, kernel, nthreads=1):
        return self._conv(self.lib.inplace_cpu_convolution, "inplace_cpu_convolution", im, kernel, nthreads)

    def convolution3DfftCUDAInPlace(self, im, kernel, device=0):
        return self._conv(self.lib.convolution3DfftCUDAInPlace, "convolution3DfftCUDAInPlace", im, kernel, device)

    def compute_quotient(self, inp, out, device=0):
        inp, out = _f32(inp), _f32(out)
        self.lib.lmvn_clear_error()
        self.lib.compute_quotient(_fp(inp), _fp(out), inp.size, int(device))
        self._check_void("compute_quotient")
        return out

    def compute_final_values(self, image, integral, weight, min_value, lam, device=0):
        image, integral, weight = _f32(image), _f32(integral), _f32(weight)
        self.lib.lmvn_clear_error()
        self.lib.compute_final_values(_fp(image), _fp(integral), _fp(weight), image.size, float(min_value), float(lam),
                                      int(device))
        self._check_void("compute_final_values")
        return image

    def iterate_fft_plain(self, inp, kernel, device=0):
        inp, kernel = _f32(inp), _f32(kernel)
        out = np.empty_like(inp)
        self.lib.lmvn_clear_error()
        self.lib.iterate_fft_plain(_fp(inp), _fp(kernel), _fp(out), C.cast(_dims(inp.shape), c_int_p),
                                   C.cast(_dims(kernel.shape), c_int_p), int(device))
        self._check_void("iterate_fft_plain")
        return out

    def iterate_fft_tikhonov(self, inp, kernel, min_value, lam, device=0):
        inp, kernel = _f32(inp), _f32(kernel)
        out = np.empty_like(inp)
        self.lib.lmvn_clear_error()
        self.lib.iterate_fft_tikhonov(_fp(inp), _fp(kernel), _fp(out), C.cast(_dims(inp.shape), c_int_p),
                                      C.cast(_dims(kernel.shape), c_int_p), inp.size, float(min_value), float(lam),
                                      int(device))
        self._check_void("iterate_fft_tikhonov")
        return out

    # -- device queries --------------------------------------------------------
    def num_devices(self) -> int:
        return int(self.lib.getNumDevicesCUDA())

    def device_name(self, dev: int) -> str:
        buf = C.create_string_buffer(256)
        self.lib.getNameDeviceCUDA(int(dev), buf)
        return buf.value.decode()

    def device_memory(self, dev: int) -> int:
        return int(self.lib.getMemDeviceCUDA(int(dev)))

    def compute_capability(self, dev: int):
        return (int(self.lib.getCUDAcomputeCapabilityMajorVersion(int(dev))),
                int(self.lib.getCUDAcomputeCapabilityMinorVersion(int(dev))))

    def select_device(self) -> int:
        return int(self.lib.selectDeviceWithHighestComputeCapability())

    # -- debug transforms --------------------------------------------------------
    def rfftn(self, a, device=-1) -> np.ndarray:
        a = _f32(a)
        nz, ny, nx = a.shape
        out = np.empty((nz, ny, nx // 2 + 1), dtype=np.complex64)
        self._check(self.lib.lmvn_debug_rfftn(_fp(a), C.cast(_dims(a.shape), c_int_p),
                                              out.ctypes.data_as(c_float_p), int(device)), "lmvn_debug_rfftn")
        return out

    def irfftn(self, spec, dims, device=-1) -> np.ndarray:
        spec = np.ascontiguousarray(spec, dtype=np.complex64)
        out = np.empty(tuple(dims), dtype=np.float32)
        self._check(self.lib.lmvn_debug_irfftn(spec.ctypes.data_as(c_float_p), C.cast(_dims(dims), c_int_p), _fp(out),
                                               int(device)), "lmvn_debug_irfftn")
        return out

    def plan(self, dims, num_views, device=-1, max_kernel_dims=None, geometry: str = "native") -> "Plan":
        return Plan(self, dims, num_views, device, max_kernel_dims, geometry)


class Plan:
    """Persistent deconvolution handle (lmvn_plan_*): views, weights and PSF spectra stay
    on the device; only psi moves."""

    def __init__(self, library: Library, dims, num_views: int, device: int = -1, max_kernel_dims=None,
                 geometry: str = "native"):
        """geometry "native": the plan works at `dims` (circular there); "embedded" / "zero": `dims` are the stack
        extents, the plan works at power-of-two extents >= dims + max_kernel_dims - 1 with periodic refill (same circular
        semantics) or zero padding (the reference GPU path's linear convolution at the borders)."""
        self.L = library
        self.dims = tuple(int(d) for d in dims)
        self.handle = C.c_void_p()
        if geometry == "native":
            library._check(library.lib.lmvn_plan_create(C.byref(self.handle), C.cast(_dims(self.dims), c_int_p),
                                                        int(num_views), int(device)), "lmvn_plan_create")
        else:
            if max_kernel_dims is None:
                raise ValueError("padded geometries need max_kernel_dims")
            fn = {"embedded": library.lib.lmvn_plan_create_embedded, "zero": library.lib.lmvn_plan_create_zero_padded}[geometry]
            library._check(fn(C.byref(self.handle), C.cast(_dims(self.dims), c_int_p),
                              C.cast(_dims(tuple(max_kernel_dims)), c_int_p), int(num_views), int(device)),
                           "lmvn_plan_create_" + geometry)

    def close(self):
        if self.handle:
            self.L.lib.lmvn_plan_destroy(self.handle)
            self.handle = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> PlanInfo:
        info = PlanInfo()
        self.L._check(self.L.lib.lmvn_plan_get_info(self.handle, C.byref(info)), "lmvn_plan_get_info")
        return info

    def set_view(self, v: int, image, weights, kernel1, kernel2):
        image, weights, kernel1, kernel2 = _f32(image), _f32(weights), _f32(kernel1), _f32(kernel2)
        if image.shape != self.dims or weights.shape != self.dims:
            raise ValueError("view / weights shape differs from the plan dims")
        self.L._check(self.L.lib.lmvn_plan_set_view(
            self.handle, int(v), _fp(image), _fp(weights), _fp(kernel1), C.cast(_dims(kernel1.shape), c_int_p),
            _fp(kernel2), C.cast(_dims(kernel2.shape), c_int_p)), "lmvn_plan_set_view")

    def set_psi(self, psi):
        psi = _f32(psi)
        if psi.shape != self.dims:
            raise ValueError("psi shape differs from the plan dims")
        self.L._check(self.L.lib.lmvn_plan_set_psi(self.handle, _fp(psi)), "lmvn_plan_set_psi")

    def get_psi(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty(self.dims, dtype=np.float32)
        out = _f32(out)
        self.L._check(self.L.lib.lmvn_plan_get_psi(self.handle, _fp(out)), "lmvn_plan_get_psi")
        return out

    def iterate(self, iterations: int, lam: float = 0.0, min_value: float = 1e-4, timed: bool = True) -> float:
        """Runs the loop on the device; returns the CUDA-event time in ms (0 if not timed)."""
        ms = C.c_float(0.0)
        self.L._check(self.L.lib.lmvn_plan_iterate(self.handle, int(iterations), float(lam), float(min_value),
                                                   C.byref(ms) if timed else None), "lmvn_plan_iterate")
        return float(ms.value)

    def convolve(self, view: int = 0, which_kernel: int = 1, repeats: int = 1) -> float:
        ms = C.c_float(0.0)
        self.L._check(self.L.lib.lmvn_plan_convolve(self.handle, int(view), int(which_kernel), int(repeats),
                                                    C.byref(ms)), "lmvn_plan_convolve")
        return float(ms.value)

    def synchronize(self):
        self.L._check(self.L.lib.lmvn_plan_synchronize(self.handle), "lmvn_plan_synchronize")

    def profile(self, lam: float = 0.0, min_value: float = 1e-4, max_entries: int = 64):
        """One (view 0, iteration) with a CUDA event after every launch.
        Returns [(kernel name, ms, algorithmic bytes)] in launch order; psi is restored."""
        names = C.create_string_buffer(48 * max_entries)
        ms = (C.c_float * max_entries)()
        nbytes = (C.c_ulonglong * max_entries)()
        count = C.c_int(0)
        self.L._check(self.L.lib.lmvn_plan_profile(self.handle, float(lam), float(min_value), max_entries, names, ms,
                                                   nbytes, C.byref(count)), "lmvn_plan_profile")
        out = []
        for i in range(count.value):
            raw = names.raw[i * 48:(i + 1) * 48]
            out.append((raw.split(b"\0", 1)[0].decode(), float(ms[i]), int(nbytes[i])))
        return out


_default: Optional[Library] = None


def load(path: Optional[str] = None) -> Library:
    """The process-wide library (built on first use if the sources are newer)."""
    global _default
    if path is not None:
        return Library(path)
    if _default is None:
        _default = Library()
    return _default
