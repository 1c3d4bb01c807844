"""lsp-dsp-units_b200 -- B200-native batched ``dspu::Convolver`` (host-side Python mirror).

Thin ctypes layer over the C ABI in ``include/b200conv.h`` (``libb200conv.so``, hand-written
sm_100a CUDA).  ``Convolver`` mirrors ``lsp::dspu::Convolver`` (reference
``include/lsp-plug.in/dsp-units/util/Convolver.h:59-113``): same method names, argument meaning
and error behaviour; ``ConvolverBatch`` is the many-instance form the engine is built for.

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible,
construction raises.  The directory name contains a hyphen, so import it through ``load()`` in
``__graft_entry__.py`` (module name ``lsp_dsp_units_b200``).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("B200CONV_LIB", os.path.join(_HERE, "libb200conv.so"))     # override: A/B builds

RANK_MIN, RANK_MAX = 8, 16
OK, ERR_ARG, ERR_NOMEM, ERR_CUDA, ERR_STATE = 0, -1, -2, -3, -4

_SZ = ctypes.c_size_t
_FP = ctypes.POINTER(ctypes.c_float)
_VP = ctypes.c_void_p


class State(ctypes.Structure):
    _fields_ = [("conv_size", _SZ), ("rank", _SZ), ("frame_size", _SZ), ("frame_off", _SZ),
                ("bins", _SZ), ("partitions", _SZ), ("part_offset", _SZ), ("frames", ctypes.c_uint64)]


class Dump(ctypes.Structure):
    """b200conv_dump_t: the 18 fields of Convolver::dump (Convolver.cpp:315-337), in its order."""
    _fields_ = ([(n, _VP) for n in ("vDataBuffer", "vFrame", "vConvBuffer", "vTaskData", "vConvData", "vDirectData")]
                + [(n, _SZ) for n in ("nDataBufferSize", "nDirectSize", "nFrameSize", "nFrameOff", "nConvSize",
                                      "nLevels", "nBlocks", "nBlocksDone", "nRank", "nBlkInit")]
                + [("fBlkCoef", ctypes.c_float), ("vData", _VP)])


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in ("launches", "frames", "h2d_bytes", "d2h_bytes",
                                               "mac_launches", "mac_algo_bytes", "mac_stream_bytes")]


class B200ConvError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("b200conv error %d: %s" % (code, text))
        self.code = code


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def build(verbose=False):
    """Compile csrc/engine.cu for sm_100a into libb200conv.so (in-tree)."""
    src = os.path.join(_HERE, "csrc", "engine.cu")
    deps = [src, os.path.join(_ROOT, "include", "b200conv.h")] + [
        os.path.join(_HERE, "csrc", h) for h in ("kernels.cuh", "equalizer.cuh", "spectral.cuh", "spectral_host.cuh",
                                                  "splitter.cuh", "matrix.cuh", "matrix_host.cuh")]
    if os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + ["-I", os.path.join(_ROOT, "include"), "-o", LIB_PATH, src]
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(" ".join(cmd))
    return LIB_PATH


_lib = None

_SIGNATURES = {
    "b200conv_create": (ctypes.c_int, [ctypes.POINTER(_VP), ctypes.c_int, _SZ]),
    "b200conv_free": (None, [_VP]),
    "b200conv_init": (ctypes.c_int, [_VP, _SZ, _FP, _SZ, _SZ, ctypes.c_float]),
    "b200conv_init_range": (ctypes.c_int, [_VP, _SZ, _FP, _SZ, _SZ, ctypes.c_float, _SZ]),
    "b200conv_init_many": (ctypes.c_int, [_VP, _SZ, ctypes.POINTER(_SZ), ctypes.POINTER(_FP), ctypes.POINTER(_SZ), _SZ,
                                          _FP, ctypes.POINTER(_SZ)]),
    "b200conv_init_shared": (ctypes.c_int, [_VP, _SZ, _SZ, ctypes.c_float]),
    "b200conv_destroy": (ctypes.c_int, [_VP, _SZ]),
    "b200conv_process": (ctypes.c_int, [_VP, ctypes.POINTER(_FP), ctypes.POINTER(_FP), _SZ]),
    "b200conv_process_planar": (ctypes.c_int, [_VP, _VP, _VP, _SZ, _SZ]),
    "b200conv_process_device": (ctypes.c_int, [_VP, _VP, _VP, _SZ, _SZ, _VP]),
    "b200conv_process_device2": (ctypes.c_int, [_VP, _VP, _SZ, _VP, _SZ, _SZ, _VP]),
    "b200conv_sync": (ctypes.c_int, [_VP]),
    "b200conv_reduce_prepare": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.c_int, ctypes.c_char_p]),
    "b200conv_reduce_connect": (ctypes.c_int, [_VP, ctypes.c_char_p]),
    "b200conv_reduce_disconnect": (ctypes.c_int, [_VP]),
    "b200conv_reduce_status": (ctypes.c_int, [_VP, ctypes.POINTER(ctypes.c_int)]),
    "b200conv_data_size": (_SZ, [_VP, _SZ]),
    "b200conv_rank": (_SZ, [_VP, _SZ]),
    "b200conv_instances": (_SZ, [_VP]),
    "b200conv_get_state": (ctypes.c_int, [_VP, _SZ, ctypes.POINTER(State)]),
    "b200conv_get_dump": (ctypes.c_int, [_VP, _SZ, ctypes.POINTER(Dump)]),
    "b200conv_get_stats": (ctypes.c_int, [_VP, ctypes.POINTER(Stats)]),
    "b200conv_reset_stats": (ctypes.c_int, [_VP]),
    "b200conv_set_profiling": (ctypes.c_int, [_VP, ctypes.c_int]),
    "b200conv_get_profile": (ctypes.c_int, [_VP, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]),
    "b200conv_stream": (_VP, [_VP]),
    "b200conv_set_option": (ctypes.c_int, [_VP, ctypes.c_char_p, ctypes.c_int]),
    "b200conv_fastconv_parse": (ctypes.c_int, [ctypes.c_int, _VP, _VP, _SZ, _SZ, _VP]),
    "b200conv_fastconv_apply": (ctypes.c_int, [ctypes.c_int, _VP, _VP, _VP, _SZ, _SZ, _VP]),
    "b200conv_fastconv_parse_apply": (ctypes.c_int, [ctypes.c_int, _VP, _VP, _VP, _SZ, _SZ, _VP]),
    "b200conv_fastconv_restore": (ctypes.c_int, [ctypes.c_int, _VP, _VP, _SZ, _SZ, _VP]),
    "b200conv_convolve": (ctypes.c_int, [ctypes.c_int, _VP, _SZ, _VP, _SZ, _VP, _SZ, _SZ, _SZ, _SZ, _VP]),
    "b200conv_linear_convolve": (ctypes.c_int, [ctypes.c_int, _VP, _SZ, _VP, _SZ, _SZ, _SZ, _VP, _SZ, _SZ]),
    "b200conv_chirp_plan": (ctypes.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, ctypes.POINTER(_SZ), _SZ, _SZ, _SZ]),
    "b200conv_chirp_linear_convolutions": (ctypes.c_int, [ctypes.c_int, _VP, _SZ, ctypes.POINTER(_FP),
                                                            ctypes.POINTER(_SZ), _SZ, _FP, _SZ, _SZ, ctypes.c_float]),
    "b200conv_eq_create": (ctypes.c_int, [ctypes.POINTER(_VP), ctypes.c_int, _SZ, _SZ]),
    "b200conv_eq_free": (None, [_VP]),
    "b200conv_eq_set_kernel": (ctypes.c_int, [_VP, _SZ, _FP, ctypes.c_int]),
    "b200conv_eq_clear": (ctypes.c_int, [_VP]),
    "b200conv_eq_process": (ctypes.c_int, [_VP, ctypes.POINTER(_FP), ctypes.POINTER(_FP), _SZ]),
    "b200conv_eq_process_planar": (ctypes.c_int, [_VP, _VP, _VP, _SZ, _SZ]),
    "b200conv_eq_process_device": (ctypes.c_int, [_VP, _VP, _SZ, _VP, _SZ, _SZ, _VP]),
    "b200conv_eq_sync": (ctypes.c_int, [_VP]),
    "b200conv_eq_stream": (_VP, [_VP]),
    "b200conv_eq_fir_size": (_SZ, [_VP]),
    "b200conv_eq_latency": (_SZ, [_VP]),
    "b200conv_eq_instances": (_SZ, [_VP]),
    "b200conv_sp_create": (ctypes.c_int, [ctypes.POINTER(_VP), ctypes.c_int, _SZ, _SZ]),
    "b200conv_sp_free": (None, [_VP]),
    "b200conv_sp_set_rank": (ctypes.c_int, [_VP, _SZ]),
    "b200conv_sp_set_phase": (ctypes.c_int, [_VP, _SZ, ctypes.c_float]),
    "b200conv_sp_bind_complex": (ctypes.c_int, [_VP, _SZ, _FP]),
    "b200conv_sp_bind_gain": (ctypes.c_int, [_VP, _SZ, _FP]),
    "b200conv_sp_unbind": (ctypes.c_int, [_VP, _SZ]),
    "b200conv_sp_process_device": (ctypes.c_int, [_VP, _VP, _SZ, _VP, _SZ, _SZ, _VP]),
    "b200conv_sp_process_planar": (ctypes.c_int, [_VP, _VP, _VP, _SZ, _SZ]),
    "b200conv_sp_reset": (ctypes.c_int, [_VP]),
    "b200conv_sp_sync": (ctypes.c_int, [_VP]),
    "b200conv_sp_stream": (_VP, [_VP]),
    "b200conv_sp_rank": (_SZ, [_VP]),
    "b200conv_sp_latency": (_SZ, [_VP]),
    "b200conv_sp_remaining": (_SZ, [_VP, _SZ]),
    "b200conv_sp_instances": (_SZ, [_VP]),
    "b200conv_ss_create": (ctypes.c_int, [ctypes.POINTER(_VP), ctypes.c_int, _SZ, _SZ, _SZ]),
    "b200conv_ss_free": (None, [_VP]),
    "b200conv_ss_set_rank": (ctypes.c_int, [_VP, _SZ]),
    "b200conv_ss_set_chunk_rank": (ctypes.c_int, [_VP, ctypes.c_long]),
    "b200conv_ss_set_phase": (ctypes.c_int, [_VP, _SZ, ctypes.c_float]),
    "b200conv_ss_bind_complex": (ctypes.c_int, [_VP, _SZ, _SZ, _FP]),
    "b200conv_ss_bind_gain": (ctypes.c_int, [_VP, _SZ, _SZ, _FP]),
    "b200conv_ss_bind_sink": (ctypes.c_int, [_VP, _SZ, _SZ]),
    "b200conv_ss_unbind": (ctypes.c_int, [_VP, _SZ, _SZ]),
    "b200conv_ss_unbind_all": (ctypes.c_int, [_VP, _SZ]),
    "b200conv_ss_bindings": (_SZ, [_VP, _SZ]),
    "b200conv_ss_process_device": (ctypes.c_int, [_VP, _VP, _SZ, _SZ, _VP, _SZ, _SZ, _VP]),
    "b200conv_ss_process_planar": (ctypes.c_int, [_VP, _VP, _VP, _SZ, _SZ]),
    "b200conv_ss_clear": (ctypes.c_int, [_VP]),
    "b200conv_ss_sync": (ctypes.c_int, [_VP]),
    "b200conv_ss_stream": (_VP, [_VP]),
    "b200conv_ss_rank": (_SZ, [_VP]),
    "b200conv_ss_chunk_rank": (_SZ, [_VP]),
    "b200conv_ss_latency": (_SZ, [_VP]),
    "b200conv_ss_instances": (_SZ, [_VP]),
    "b200conv_ss_handlers": (_SZ, [_VP]),
    "b200conv_mx_create": (ctypes.c_int, [ctypes.POINTER(_VP), ctypes.c_int, _SZ, _SZ, _SZ]),
    "b200conv_mx_free": (None, [_VP]),
    "b200conv_mx_set_routes": (ctypes.c_int, [_VP, _SZ, ctypes.POINTER(_SZ), ctypes.POINTER(_SZ), ctypes.POINTER(_FP),
                                              ctypes.POINTER(_SZ)]),
    "b200conv_mx_set_irs": (ctypes.c_int, [_VP, _SZ, ctypes.POINTER(_SZ), ctypes.POINTER(_FP), ctypes.POINTER(_SZ),
                                           _SZ, _VP]),
    "b200conv_mx_fade_remaining": (_SZ, [_VP]),
    "b200conv_mx_clear": (ctypes.c_int, [_VP]),
    "b200conv_mx_process_device": (ctypes.c_int, [_VP, _VP, _SZ, _VP, _SZ, _SZ, _VP]),
    "b200conv_mx_process_planar": (ctypes.c_int, [_VP, _VP, _SZ, _VP, _SZ, _SZ]),
    "b200conv_mx_sync": (ctypes.c_int, [_VP]),
    "b200conv_mx_stream": (_VP, [_VP]),
    "b200conv_mx_inputs": (_SZ, [_VP]),
    "b200conv_mx_outputs": (_SZ, [_VP]),
    "b200conv_mx_rank": (_SZ, [_VP]),
    "b200conv_mx_frame_size": (_SZ, [_VP]),
    "b200conv_mx_routes": (_SZ, [_VP]),
    "b200conv_last_error": (ctypes.c_char_p, []),
    "b200conv_version": (ctypes.c_char_p, []),
}


def lib():
    """The loaded C-ABI library.  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                "%s is missing: build it with __graft_entry__.build() (nvcc, sm_100a). "
                "This engine has no CPU fallback." % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def _check(rc):
    if rc != OK:
        raise B200ConvError(rc, lib().b200conv_last_error().decode())


def _ptr(a):
    return a.ctypes.data_as(_FP)


class ConvolverBatch:
    """``instances`` independent convolvers on one GPU, advanced together (include/b200conv.h)."""

    def __init__(self, instances, device=-1):
        self._h = _VP()
        _check(lib().b200conv_create(ctypes.byref(self._h), device, instances))
        self.instances = instances

    # -- Convolver::init / destroy ------------------------------------------------------------
    def init(self, idx, data, rank, phase=0.0, part_offset=0):
        """``Convolver::init(data, count, rank, phase)`` for instance ``idx``; True on success,
        False only on allocation failure (previous state kept), like the reference."""
        data = np.ascontiguousarray(data, dtype=np.float32)
        rc = lib().b200conv_init_range(self._h, idx, _ptr(data), data.size, rank, phase, part_offset)
        if rc == ERR_NOMEM:
            return False
        _check(rc)
        return True

    def init_many(self, indices, irs, rank, phases=None, part_offsets=None):
        """``Convolver::init`` for many instances in one call (one allocation, one upload, one
        transform launch); an empty IR destroys its instance.  False on allocation failure."""
        irs = [np.ascontiguousarray(x, dtype=np.float32) for x in irs]
        n = len(indices)
        assert len(irs) == n
        ph = (ctypes.c_float * n)(*(phases if phases is not None else [0.0] * n))
        po = (_SZ * n)(*(part_offsets if part_offsets is not None else [0] * n))
        rc = lib().b200conv_init_many(self._h, n, (_SZ * n)(*indices), (_FP * n)(*[_ptr(x) for x in irs]),
                                      (_SZ * n)(*[x.size for x in irs]), rank, ph, po)
        if rc == ERR_NOMEM:
            return False
        _check(rc)
        return True

    def init_shared(self, idx, src_idx, phase=0.0):
        """Instance ``idx`` gets the same impulse response as ``src_idx`` and shares its device spectra."""
        rc = lib().b200conv_init_shared(self._h, idx, src_idx, phase)
        if rc == ERR_NOMEM:
            return False
        _check(rc)
        return True

    def destroy(self, idx):
        _check(lib().b200conv_destroy(self._h, idx))

    # -- Convolver::process -------------------------------------------------------------------
    def process(self, src, out=None):
        """Host arrays ``[instances][count]`` float32 (rows are the planar per-instance buffers).

        Row-contiguous 2-D arrays go through ``b200conv_process_planar`` (one strided copy each
        way); anything else through the per-instance pointer table of ``b200conv_process``."""
        src = np.asarray(src, dtype=np.float32)
        if src.ndim == 1:
            src = src[None, :]
        assert src.shape[0] == self.instances
        if out is None:
            out = np.empty(src.shape, dtype=np.float32)
        elif (not isinstance(out, np.ndarray) or out.dtype != np.float32 or out.shape != src.shape
              or not out.flags.writeable):
            # the C ABI reinterprets the buffer as float*: anything else would be silent garbage
            raise ValueError("out must be a writeable float32 array of shape %r" % (src.shape,))
        n = src.shape[1]
        planar = (src.strides[1] == 4 and out.strides[1] == 4 and out.shape == src.shape
                  and (self.instances == 1 or (src.strides[0] == out.strides[0] and src.strides[0] % 4 == 0
                                               and src.strides[0] >= 4 * n)))
        if planar:
            stride = (src.strides[0] // 4) if self.instances > 1 else n
            _check(lib().b200conv_process_planar(self._h, out.ctypes.data, src.ctypes.data, stride, n))
            return out
        src = np.ascontiguousarray(src)
        tmp = out if out.flags.c_contiguous else np.empty(src.shape, dtype=np.float32)
        srcs = (_FP * self.instances)(*[_ptr(src[i]) for i in range(self.instances)])
        dsts = (_FP * self.instances)(*[_ptr(tmp[i]) for i in range(self.instances)])
        _check(lib().b200conv_process(self._h, dsts, srcs, n))
        if tmp is not out:
            out[...] = tmp
        return out

    def process_pointers(self, dsts, srcs, count):
        """``b200conv_process`` with explicit per-instance host arrays (any alignment)."""
        sp = (_FP * self.instances)(*[_ptr(a) for a in srcs])
        dp = (_FP * self.instances)(*[_ptr(a) for a in dsts])
        _check(lib().b200conv_process(self._h, dp, sp, count))

    def process_device(self, dst_ptr, src_ptr, stride, count, stream=None, dst_stride=None):
        """Device pointers (ints), ``[instances][stride]`` floats; asynchronous.  ``dst_stride``
        (default: ``stride``) lets the output matrix have its own row pitch."""
        _check(lib().b200conv_process_device2(self._h, dst_ptr, stride if dst_stride is None else dst_stride,
                                              src_ptr, stride, count, stream))

    def sync(self):
        _check(lib().b200conv_sync(self._h))

    # -- partition-range sharding: fused NVLink reduce (see include/b200conv.h) -----------------
    def reduce_prepare(self, grank, world):
        """Allocates the exchange buffer; returns its 64-byte CUDA IPC handle."""
        buf = ctypes.create_string_buffer(64)
        _check(lib().b200conv_reduce_prepare(self._h, grank, world, buf))
        return buf.raw

    def reduce_connect(self, handles):
        """``handles``: the IPC handles of all ranks, in rank order."""
        _check(lib().b200conv_reduce_connect(self._h, b"".join(handles)))

    def reduce_disconnect(self):
        _check(lib().b200conv_reduce_disconnect(self._h))

    def reduce_timed_out(self):
        flag = ctypes.c_int(0)
        _check(lib().b200conv_reduce_status(self._h, ctypes.byref(flag)))
        return bool(flag.value)

    # -- queries ------------------------------------------------------------------------------
    def data_size(self, idx):
        return int(lib().b200conv_data_size(self._h, idx))

    def rank(self, idx):
        return int(lib().b200conv_rank(self._h, idx))

    def state(self, idx):
        st = State()
        _check(lib().b200conv_get_state(self._h, idx, ctypes.byref(st)))
        return {n: int(getattr(st, n)) for n, _ in State._fields_}

    def dump(self, idx):
        """The fields ``Convolver::dump`` writes, as a dict in the reference's order."""
        d = Dump()
        _check(lib().b200conv_get_dump(self._h, idx, ctypes.byref(d)))
        return {n: getattr(d, n) for n, _ in Dump._fields_}

    def stats(self):
        st = Stats()
        _check(lib().b200conv_get_stats(self._h, ctypes.byref(st)))
        return {n: int(getattr(st, n)) for n, _ in Stats._fields_}

    def reset_stats(self):
        _check(lib().b200conv_reset_stats(self._h))

    def set_profiling(self, enable):
        _check(lib().b200conv_set_profiling(self._h, int(bool(enable))))

    def profile(self):
        """(summed k_mac device time in ms, k_mac launches) since the last call."""
        ms, n = ctypes.c_double(0.0), ctypes.c_uint64(0)
        _check(lib().b200conv_get_profile(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, int(n.value)

    def stream(self):
        return lib().b200conv_stream(self._h)

    def set_option(self, name, value):
        """Tuning / A-B knobs, see b200conv_set_option in include/b200conv.h."""
        _check(lib().b200conv_set_option(self._h, name.encode(), int(value)))

    def close(self):
        if self._h:
            lib().b200conv_free(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Convolver:
    """Mirror of ``lsp::dspu::Convolver``: a batch of one (Convolver.h:59-113)."""

    def __init__(self, device=-1):
        self._device = device
        self._b = None

    def init(self, data, rank, phase=0.0):
        data = np.ascontiguousarray(data, dtype=np.float32)
        if data.size == 0:                      # Convolver.cpp:80-84
            self.destroy()
            return True
        fresh = ConvolverBatch(1, self._device)
        if not fresh.init(0, data, rank, phase):
            fresh.close()
            return False                        # previous state intact (Convolver.cpp:103-108)
        self.destroy()
        self._b = fresh
        return True

    def destroy(self):
        if self._b is not None:
            self._b.close()
            self._b = None

    def process(self, src, out=None):
        src = np.ascontiguousarray(src, dtype=np.float32)
        if out is None:
            out = np.empty_like(src)
        elif (not isinstance(out, np.ndarray) or out.dtype != np.float32 or out.shape != src.shape
              or not out.flags.writeable):
            raise ValueError("out must be a writeable float32 array of shape %r" % (src.shape,))
        if self._b is None:                     # Convolver.cpp:219-223
            out[...] = 0.0
            return out
        if src.size:
            self._b.process(src[None, :], out[None, :])
        return out

    def run(self, src, step):
        """Feed ``src`` in calls of ``step`` samples (reference utest helper convolver.cpp:43-53)."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        out = np.zeros_like(src)
        for i in range(0, src.size, step):
            self.process(src[i:i + step], out[i:i + step])
        return out

    def data_size(self):
        return self._b.data_size(0) if self._b is not None else 0

    def rank(self):
        return self._b.rank(0) if self._b is not None else 0

    def state(self):
        return self._b.state(0) if self._b is not None else None


def linear_convolve(src, h, rank=11, device=0):
    """Full linear convolution of every row of ``src`` with ``h`` on the GPU
    (``b200conv_linear_convolve``; SyncChirpProcessor::do_linear_convolution's operation)."""
    src = np.ascontiguousarray(src, dtype=np.float32)
    one = src.ndim == 1
    if one:
        src = src[None, :]
    h = np.ascontiguousarray(h, dtype=np.float32)
    count, nx = src.shape
    out = np.empty((count, nx + h.size - 1), dtype=np.float32)
    _check(lib().b200conv_linear_convolve(device, out.ctypes.data, out.shape[1], src.ctypes.data, nx, nx,
                                          count, h.ctypes.data, h.size, rank))
    return out[0] if one else out


class ChirpPlan(ctypes.Structure):
    _fields_ = [(n, _SZ) for n in ("partition_size", "conv_rank", "image", "allocation_size")]


def chirp_plan(in_len, inverse_len, part_size_limit):
    """``calculateConvolutionPartitionSize`` + ``calculateConvolutionParameters``
    (SyncChirpProcessor.cpp:1224-1250, 1299-1331); no device needed."""
    n = len(in_len)
    plan = ChirpPlan()
    arrs = [(_SZ * n)() for _ in range(5)]
    _check(lib().b200conv_chirp_plan(ctypes.byref(plan), *[ctypes.cast(a, _VP) for a in arrs],
                                     (_SZ * n)(*in_len), n, inverse_len, part_size_limit))
    out = {k: int(getattr(plan, k)) for k, _ in ChirpPlan._fields_}
    for k, a in zip(("partitions", "padded", "prepends", "conv_lengths", "align_offsets"), arrs):
        out[k] = list(a)
    return out


def chirp_linear_convolutions(inputs, inverse, part_size_limit=0, scale=1.0, device=0):
    """``SyncChirpProcessor::do_linear_convolutions`` on plain arrays: ``inputs[ch]`` is channel
    ``ch``'s recording from its offset on; returns ``[nchannels][allocation_size]`` float32."""
    inputs = [np.ascontiguousarray(x, dtype=np.float32) for x in inputs]
    inverse = np.ascontiguousarray(inverse, dtype=np.float32)
    n = len(inputs)
    lens = [x.size for x in inputs]
    plan = chirp_plan(lens, inverse.size, part_size_limit)
    res = np.empty((n, plan["allocation_size"]), dtype=np.float32)
    _check(lib().b200conv_chirp_linear_convolutions(
        device, res.ctypes.data, res.shape[1], (_FP * n)(*[_ptr(x) for x in inputs]), (_SZ * n)(*lens), n,
        _ptr(inverse), inverse.size, part_size_limit, scale))
    return res


class EqualizerBatch:
    """Data path of ``dspu::Equalizer`` (EQM_FIR / EQM_FFT) for ``instances`` equalizers on one GPU
    (``b200conv_eq_*``): ``set_kernel`` takes the finished ``2**fir_rank``-tap impulse response,
    ``process`` has ``fir_size`` samples of latency (reference Equalizer.cpp:474-518)."""

    def __init__(self, instances, fir_rank, device=-1):
        self._h = _VP()
        _check(lib().b200conv_eq_create(ctypes.byref(self._h), device, instances, fir_rank))
        self.instances = instances
        self.fir_size = lib().b200conv_eq_fir_size(self._h)

    def close(self):
        if self._h:
            lib().b200conv_eq_free(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def latency(self):
        return lib().b200conv_eq_latency(self._h)

    def set_kernel(self, idx, ir, smooth=False):
        ir = np.ascontiguousarray(ir, dtype=np.float32)
        if ir.size != self.fir_size:
            raise ValueError("kernel must hold fir_size = %d taps" % self.fir_size)
        _check(lib().b200conv_eq_set_kernel(self._h, idx, _ptr(ir), int(bool(smooth))))

    def clear(self):
        _check(lib().b200conv_eq_clear(self._h))

    def process(self, src):
        """src: [instances][samples] float32 (host) -> same shape."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        if src.ndim != 2 or src.shape[0] != self.instances:
            raise ValueError("expected [instances][samples]")
        out = np.empty_like(src)
        _check(lib().b200conv_eq_process_planar(self._h, out.ctypes.data, src.ctypes.data, src.shape[1],
                                                src.shape[1]))
        return out

    def process_pointers(self, dsts, srcs, samples):
        n = self.instances
        d = (_FP * n)(*[_ptr(a) for a in dsts])
        s = (_FP * n)(*[_ptr(a) for a in srcs])
        _check(lib().b200conv_eq_process(self._h, d, s, samples))

    def process_device(self, dst_ptr, dst_stride, src_ptr, src_stride, samples, stream=None):
        _check(lib().b200conv_eq_process_device(self._h, dst_ptr, dst_stride, src_ptr, src_stride, samples,
                                                stream))

    def sync(self):
        _check(lib().b200conv_eq_sync(self._h))

    def stream(self):
        return lib().b200conv_eq_stream(self._h)


class SpectralProcessorBatch:
    """``instances`` x ``lsp::dspu::SpectralProcessor`` on one GPU (``b200conv_sp_*``): same method
    names and meaning as the reference class; the host callback of the reference is replaced by a
    per-instance spectral table (``bind_complex`` / ``bind_gain``)."""

    def __init__(self, instances, max_rank, device=-1):
        self._h = _VP()
        _check(lib().b200conv_sp_create(ctypes.byref(self._h), device, instances, max_rank))
        self.instances = instances

    def close(self):
        if self._h:
            lib().b200conv_sp_free(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rank(self, rank):
        _check(lib().b200conv_sp_set_rank(self._h, rank))

    def set_phase(self, idx, phase):
        _check(lib().b200conv_sp_set_phase(self._h, idx, phase))

    def get_rank(self):
        return int(lib().b200conv_sp_rank(self._h))

    def latency(self):
        return int(lib().b200conv_sp_latency(self._h))

    def remaining(self, idx):
        return int(lib().b200conv_sp_remaining(self._h, idx))

    def bind_complex(self, idx, table):
        t = np.ascontiguousarray(table, dtype=np.complex64).view(np.float32)
        if t.size != 2 << self.get_rank():
            raise ValueError("table must hold 2**rank complex bins")
        _check(lib().b200conv_sp_bind_complex(self._h, idx, _ptr(t)))

    def bind_gain(self, idx, gain):
        g = np.ascontiguousarray(gain, dtype=np.float32)
        if g.size != 1 << self.get_rank():
            raise ValueError("gain must hold 2**rank values")
        _check(lib().b200conv_sp_bind_gain(self._h, idx, _ptr(g)))

    def unbind(self, idx):
        _check(lib().b200conv_sp_unbind(self._h, idx))

    def reset(self):
        _check(lib().b200conv_sp_reset(self._h))

    def process(self, src):
        """src: [instances][samples] float32 (host) -> same shape (synchronous)."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        if src.ndim != 2 or src.shape[0] != self.instances:
            raise ValueError("expected [instances][samples]")
        out = np.empty_like(src)
        _check(lib().b200conv_sp_process_planar(self._h, out.ctypes.data, src.ctypes.data, src.shape[1], src.shape[1]))
        return out

    def process_device(self, dst_ptr, dst_stride, src_ptr, src_stride, samples, stream=None):
        _check(lib().b200conv_sp_process_device(self._h, dst_ptr, dst_stride, src_ptr, src_stride, samples, stream))

    def sync(self):
        _check(lib().b200conv_sp_sync(self._h))

    def stream(self):
        return lib().b200conv_sp_stream(self._h)


class SpectralSplitterBatch:
    """``instances`` x ``lsp::dspu::SpectralSplitter`` on one GPU (``b200conv_ss_*``): same method names
    and meaning as the reference class; the host callbacks of the reference are replaced per handler
    by a spectral table (``bind_complex`` / ``bind_gain`` -- the latter is ``FFTCrossover``'s band) or by
    nothing (``bind_sink``), and the sink of handler ``h`` is row ``h`` of the output."""

    def __init__(self, instances, max_rank, handlers, device=-1):
        self._h = _VP()
        _check(lib().b200conv_ss_create(ctypes.byref(self._h), device, instances, max_rank, handlers))
        self.instances = instances
        self.handlers = handlers

    def close(self):
        if self._h:
            lib().b200conv_ss_free(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rank(self, rank):
        _check(lib().b200conv_ss_set_rank(self._h, rank))

    def set_chunk_rank(self, rank):
        _check(lib().b200conv_ss_set_chunk_rank(self._h, rank))

    def set_phase(self, idx, phase):
        _check(lib().b200conv_ss_set_phase(self._h, idx, phase))

    def rank(self):
        return int(lib().b200conv_ss_rank(self._h))

    def chunk_rank(self):
        return int(lib().b200conv_ss_chunk_rank(self._h))

    def latency(self):
        return int(lib().b200conv_ss_latency(self._h))

    def bindings(self, idx):
        return int(lib().b200conv_ss_bindings(self._h, idx))

    def bind_complex(self, idx, handler, table):
        t = np.ascontiguousarray(table, dtype=np.complex64).view(np.float32)
        if t.size != 2 << self.rank():
            raise ValueError("table must hold 2**rank complex bins")
        _check(lib().b200conv_ss_bind_complex(self._h, idx, handler, _ptr(t)))

    def bind_gain(self, idx, handler, gain):
        g = np.ascontiguousarray(gain, dtype=np.float32)
        if g.size != 1 << self.rank():
            raise ValueError("gain must hold 2**rank values")
        _check(lib().b200conv_ss_bind_gain(self._h, idx, handler, _ptr(g)))

    def bind_sink(self, idx, handler):
        _check(lib().b200conv_ss_bind_sink(self._h, idx, handler))

    def unbind(self, idx, handler):
        _check(lib().b200conv_ss_unbind(self._h, idx, handler))

    def unbind_all(self, idx):
        _check(lib().b200conv_ss_unbind_all(self._h, idx))

    def clear(self):
        _check(lib().b200conv_ss_clear(self._h))

    def process(self, src):
        """src: [instances][samples] float32 (host) -> [handlers][instances][samples] (synchronous);
        rows of handlers that are not bound stay zero."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        if src.ndim != 2 or src.shape[0] != self.instances:
            raise ValueError("expected [instances][samples]")
        out = np.zeros((self.handlers,) + src.shape, dtype=np.float32)
        _check(lib().b200conv_ss_process_planar(self._h, out.ctypes.data, src.ctypes.data, src.shape[1], src.shape[1]))
        return out

    def process_device(self, dst_ptr, band_stride, dst_stride, src_ptr, src_stride, samples, stream=None):
        _check(lib().b200conv_ss_process_device(self._h, dst_ptr, band_stride, dst_stride, src_ptr, src_stride, samples, stream))

    def sync(self):
        _check(lib().b200conv_ss_sync(self._h))

    def stream(self):
        return lib().b200conv_ss_stream(self._h)


class MatrixConvolver:
    """``inputs`` x ``outputs`` matrix of routed convolutions on one GPU (``b200conv_mx_*``): output ``o``
    is the sum, over the routes ``(i, o, ir)``, of input ``i`` convolved with ``ir``.  One spectrum ring
    per input and one inverse transform per output, whatever the number of routes.  Calls must bring
    whole frames (a multiple of ``frame_size()`` samples)."""

    def __init__(self, inputs, outputs, rank, device=-1):
        self._h = _VP()
        _check(lib().b200conv_mx_create(ctypes.byref(self._h), device, inputs, outputs, rank))
        self.inputs = inputs
        self.outputs = outputs
        self.rank = rank

    def close(self):
        if self._h:
            lib().b200conv_mx_free(self._h)
            self._h = _VP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_routes(self, routes):
        """``routes``: ``[(input, output, ir), ...]``; replaces the routing and discards the history."""
        routes = list(routes)
        n = len(routes)
        irs = [np.ascontiguousarray(h, dtype=np.float32) for _, _, h in routes]
        _check(lib().b200conv_mx_set_routes(self._h, n, (_SZ * n)(*[int(r[0]) for r in routes]),
                                            (_SZ * n)(*[int(r[1]) for r in routes]),
                                            (_FP * n)(*[_ptr(h) for h in irs]), (_SZ * n)(*[h.size for h in irs])))

    def set_irs(self, changes, fade=0, stream=None):
        """``changes``: ``[(route, ir), ...]`` with ``route`` the index in the last ``set_routes``.  Keeps the
        input history and crossfades each changed route from its old IR to the new one over ``fade``
        samples, starting with the next call (0: a hard switch).  Stream-ordered like ``process_device``
        (``stream`` None = the object's own stream); does not wait for the device."""
        changes = list(changes)
        n = len(changes)
        irs = [np.ascontiguousarray(h, dtype=np.float32).ravel() for _, h in changes]
        _check(lib().b200conv_mx_set_irs(self._h, n, (_SZ * n)(*[int(c[0]) for c in changes]),
                                         (_FP * n)(*[_ptr(h) for h in irs]), (_SZ * n)(*[h.size for h in irs]),
                                         int(fade), stream))

    def fade_remaining(self):
        """Samples of the crossfade not yet covered by the calls enqueued so far (0: none running)."""
        return int(lib().b200conv_mx_fade_remaining(self._h))

    def clear(self):
        _check(lib().b200conv_mx_clear(self._h))

    def process(self, src):
        """src: [inputs][n] float32 (host) -> [outputs][n] (synchronous)."""
        src = np.ascontiguousarray(src, dtype=np.float32)
        if src.ndim != 2 or src.shape[0] != self.inputs:
            raise ValueError("expected [inputs][samples]")
        n = src.shape[1]
        out = np.empty((self.outputs, n), dtype=np.float32)
        _check(lib().b200conv_mx_process_planar(self._h, out.ctypes.data, n, src.ctypes.data, n, n))
        return out

    def process_device(self, dst_ptr, dst_stride, src_ptr, src_stride, n, stream=None):
        """Device pointers (ints): ``src`` [inputs][src_stride], ``dst`` [outputs][dst_stride] floats;
        stream-ordered (``stream`` None = the object's own stream)."""
        _check(lib().b200conv_mx_process_device(self._h, dst_ptr, dst_stride, src_ptr, src_stride, n, stream))

    def sync(self):
        _check(lib().b200conv_mx_sync(self._h))

    def stream(self):
        return lib().b200conv_mx_stream(self._h)

    def frame_size(self):
        return int(lib().b200conv_mx_frame_size(self._h))

    def routes(self):
        return int(lib().b200conv_mx_routes(self._h))
