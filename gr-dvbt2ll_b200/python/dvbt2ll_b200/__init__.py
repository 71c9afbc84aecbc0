"""dvbt2ll_b200 -- Python face of libdvbt2ll_cuda.so (ctypes over the C ABI in include/dvbt2ll_cuda.h).

Mirrors the reference's Python surface (python/__init__.py:27-31 re-exports the SWIG module: the enum
constants plus one factory per block, e.g. ``dvbt2ll.bbheaderbch_bb(framesize, rate, mode, inband,
fecblocks, tsrate)``) with the same factory names, argument order and meaning.  Instead of being wired
into a GNU Radio flowgraph the returned objects expose ``work()`` -- the block's general_work() on
host buffers -- so the parity tests can drive them exactly like the reference blocks.

There is no CPU fallback: work() raises if the CUDA library or a device is missing.
"""
import ctypes as C
import os

import numpy as np

from .configs import *  # noqa: F401,F403  (enum constants, CONFIGS, make_ts)
from . import configs

_HERE = os.path.dirname(os.path.abspath(__file__))
# DVBT2LL_LIB selects another build of the same library (A/B timing of kernel variants, the bounds-checking debug build)
LIB_PATH = os.environ.get("DVBT2LL_LIB") or os.path.normpath(os.path.join(_HERE, "..", "..", "libdvbt2ll_cuda.so"))

_lib = None

EXPORTED_SYMBOLS = [
    "dvbt2ll_last_error", "dvbt2ll_version", "dvbt2ll_kernel_launches", "dvbt2ll_device_available",
    "dvbt2ll_output_multiple", "dvbt2ll_forecast", "dvbt2ll_work", "dvbt2ll_work_device", "dvbt2ll_warnings",
    "dvbt2ll_destroy", "dvbt2ll_plan_get", "dvbt2ll_bbheaderbch_create", "dvbt2ll_ldpc_create",
    "dvbt2ll_interleavermod_create", "dvbt2ll_framemapperfint_create", "dvbt2ll_pilotgenp1insert_create",
    "dvbt2ll_chain_create", "dvbt2ll_chain_ts_bytes_per_frame", "dvbt2ll_chain_ts_bytes", "dvbt2ll_chain_samples_per_frame",
    "dvbt2ll_chain_fecframes_per_frame", "dvbt2ll_chain_run_device", "dvbt2ll_chain_run_host",
    "dvbt2ll_chain_tap", "dvbt2ll_chain_stage_ms", "dvbt2ll_chain_enable_timing", "dvbt2ll_chain_set_sink",
    "dvbt2ll_set_overfull_policy", "dvbt2ll_set_host_register", "dvbt2ll_link", "dvbt2ll_link_hits", "dvbt2ll_link_lazy_host", "dvbt2ll_link_late_writes", "dvbt2ll_set_auto_link",
    "dvbt2ll_gather_last_error", "dvbt2ll_gather_create", "dvbt2ll_gather_export", "dvbt2ll_gather_connect",
    "dvbt2ll_gather_acquire", "dvbt2ll_gather_push", "dvbt2ll_gather_wait", "dvbt2ll_gather_release",
    "dvbt2ll_gather_side_stream", "dvbt2ll_gather_destroy",
    "dvbt2ll_copy_to_host", "dvbt2ll_copy_to_device", "dvbt2ll_device_alloc", "dvbt2ll_device_free",
    "dvbt2ll_device_count", "dvbt2ll_set_device", "dvbt2ll_device_synchronize",
    "dvbt2ll_stream_create", "dvbt2ll_stream_destroy", "dvbt2ll_stream_synchronize",
    "dvbt2ll_chain_create_multiplp", "dvbt2ll_chain_num_plp", "dvbt2ll_chain_plp_ts_bytes",
    "dvbt2ll_chain_history_bytes", "dvbt2ll_ts_sync", "dvbt2ll_ts_fill", "dvbt2ll_chain_create_plps",
    "dvbt2ll_chain_set_papr_tr", "dvbt2ll_chain_set_miso", "dvbt2ll_chain_run_device_miso", "dvbt2ll_chain_run_host_miso",
]
GATHER_BLOB_BYTES = 256


class ChainParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "framesize", "rate", "constellation", "rotation", "fecblocks", "tiblocks", "carriermode", "fftsize",
        "guardinterval", "l1constellation", "pilotpattern", "t2frames", "numdatasyms", "paprmode", "version",
        "preamble", "inputmode", "reservedbiasbits", "l1scrambled", "inband", "misogroup", "equalization",
        "bandwidth", "vlength", "tsrate")]


class PlpParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("fecblocks", "framesize", "rate", "constellation", "rotation")]


PLP_KEYS = ("framesize", "rate", "constellation", "rotation")


def plp_params(cfg):
    """cfg["plps"] with every PLP's missing framesize / rate / constellation / rotation taken from the cfg."""
    return [dict({k: int(cfg[k]) for k in PLP_KEYS}, **{k: int(v) for k, v in p.items()}) for p in cfg["plps"]]


def lib():
    """Load libdvbt2ll_cuda.so (built in-tree by gr-dvbt2ll_b200/csrc/Makefile); raises if missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libdvbt2ll_cuda.so not built: run `make -C gr-dvbt2ll_b200/csrc` "
                               "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        vp, ci, cll = C.c_void_p, C.c_int, C.c_longlong
        L.dvbt2ll_last_error.restype = C.c_char_p
        L.dvbt2ll_version.restype = C.c_char_p
        L.dvbt2ll_kernel_launches.restype = cll
        L.dvbt2ll_output_multiple.argtypes = [vp]
        L.dvbt2ll_forecast.argtypes = [vp, ci]
        L.dvbt2ll_work.argtypes = [vp, vp, ci, vp, ci, C.POINTER(ci)]
        L.dvbt2ll_work_device.argtypes = [vp, vp, ci, vp, ci, C.POINTER(ci), vp]
        L.dvbt2ll_warnings.argtypes = [vp]
        L.dvbt2ll_destroy.argtypes = [vp]
        L.dvbt2ll_plan_get.restype = cll
        L.dvbt2ll_plan_get.argtypes = [vp, C.c_char_p, vp, cll]
        for name, n in (("dvbt2ll_bbheaderbch_create", 6), ("dvbt2ll_ldpc_create", 2),
                        ("dvbt2ll_interleavermod_create", 4), ("dvbt2ll_framemapperfint_create", 20),
                        ("dvbt2ll_pilotgenp1insert_create", 12)):
            f = getattr(L, name)
            f.restype = vp
            f.argtypes = [ci] * n
        L.dvbt2ll_chain_create.restype = vp
        L.dvbt2ll_chain_create.argtypes = [C.POINTER(ChainParams), ci, ci]
        L.dvbt2ll_chain_ts_bytes_per_frame.restype = cll
        L.dvbt2ll_chain_ts_bytes_per_frame.argtypes = [vp]
        L.dvbt2ll_chain_ts_bytes.restype = cll
        L.dvbt2ll_chain_ts_bytes.argtypes = [vp, cll, ci]
        L.dvbt2ll_chain_samples_per_frame.restype = cll
        L.dvbt2ll_chain_samples_per_frame.argtypes = [vp]
        L.dvbt2ll_chain_fecframes_per_frame.argtypes = [vp]
        L.dvbt2ll_chain_run_device.argtypes = [vp, vp, cll, ci, ci, cll, vp, vp]
        L.dvbt2ll_chain_run_host.argtypes = [vp, vp, cll, ci, ci, cll, vp]
        L.dvbt2ll_chain_tap.restype = cll
        L.dvbt2ll_chain_tap.argtypes = [vp, C.c_char_p, vp, cll]
        L.dvbt2ll_chain_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.dvbt2ll_chain_enable_timing.argtypes = [vp, ci]
        L.dvbt2ll_chain_set_sink.argtypes = [vp, ci, C.c_float]
        L.dvbt2ll_chain_set_papr_tr.argtypes = [vp, ci, C.c_float, C.c_float]
        L.dvbt2ll_chain_set_miso.argtypes = [vp, ci]
        L.dvbt2ll_chain_run_device_miso.argtypes = [vp, vp, cll, ci, ci, cll, vp, vp, vp]
        L.dvbt2ll_chain_run_host_miso.argtypes = [vp, vp, cll, ci, ci, cll, vp, vp]
        L.dvbt2ll_set_overfull_policy.argtypes = [ci]
        L.dvbt2ll_set_overfull_policy.restype = None
        L.dvbt2ll_set_host_register.argtypes = [vp, ci]
        L.dvbt2ll_set_host_register.restype = None
        L.dvbt2ll_link.argtypes = [vp, vp]
        L.dvbt2ll_link_hits.argtypes = [vp]
        L.dvbt2ll_link_hits.restype = cll
        L.dvbt2ll_link_lazy_host.argtypes = [vp, ci]
        L.dvbt2ll_set_auto_link.argtypes = [ci]
        L.dvbt2ll_set_auto_link.restype = None
        L.dvbt2ll_link_late_writes.argtypes = [vp]
        L.dvbt2ll_link_late_writes.restype = cll
        sz = C.c_size_t
        L.dvbt2ll_gather_last_error.restype = C.c_char_p
        L.dvbt2ll_gather_create.restype = vp
        L.dvbt2ll_gather_create.argtypes = [ci, ci, ci, ci, sz, sz, ci]
        L.dvbt2ll_gather_export.argtypes = [vp, vp, sz]
        L.dvbt2ll_gather_connect.argtypes = [vp, vp, sz]
        L.dvbt2ll_gather_acquire.argtypes = [vp, cll, sz, vp, C.POINTER(vp)]
        L.dvbt2ll_gather_push.argtypes = [vp, cll, sz, sz, vp]
        L.dvbt2ll_gather_wait.argtypes = [vp, cll, vp, C.POINTER(vp)]
        L.dvbt2ll_gather_release.argtypes = [vp, cll, vp]
        L.dvbt2ll_gather_side_stream.restype = vp
        L.dvbt2ll_gather_side_stream.argtypes = [vp]
        L.dvbt2ll_gather_destroy.argtypes = [vp]
        L.dvbt2ll_gather_destroy.restype = None
        L.dvbt2ll_copy_to_host.argtypes = [vp, vp, sz]
        L.dvbt2ll_copy_to_device.argtypes = [vp, vp, sz]
        L.dvbt2ll_device_alloc.restype = vp
        L.dvbt2ll_device_alloc.argtypes = [sz]
        L.dvbt2ll_device_free.argtypes = [vp]
        L.dvbt2ll_device_free.restype = None
        L.dvbt2ll_set_device.argtypes = [ci]
        L.dvbt2ll_stream_create.restype = vp
        L.dvbt2ll_stream_destroy.argtypes = [vp]
        L.dvbt2ll_stream_destroy.restype = None
        L.dvbt2ll_stream_synchronize.argtypes = [vp]
        L.dvbt2ll_chain_create_multiplp.restype = vp
        L.dvbt2ll_chain_create_multiplp.argtypes = [C.POINTER(ChainParams), ci, C.POINTER(ci), ci, ci]
        L.dvbt2ll_chain_num_plp.argtypes = [vp]
        L.dvbt2ll_chain_create_plps.restype = vp
        L.dvbt2ll_chain_create_plps.argtypes = [C.POINTER(ChainParams), ci, C.POINTER(PlpParams), ci, ci]
        L.dvbt2ll_chain_plp_ts_bytes.restype = cll
        L.dvbt2ll_chain_plp_ts_bytes.argtypes = [vp, ci, cll, ci]
        L.dvbt2ll_chain_history_bytes.restype = cll
        L.dvbt2ll_chain_history_bytes.argtypes = [vp, cll]
        L.dvbt2ll_ts_sync.restype = cll
        L.dvbt2ll_ts_sync.argtypes = [vp, sz]
        L.dvbt2ll_ts_fill.restype = cll
        L.dvbt2ll_ts_fill.argtypes = [vp, sz, vp, sz, cll]
        _lib = L
    return _lib


def last_error():
    return lib().dvbt2ll_last_error().decode()


def device_available():
    return bool(lib().dvbt2ll_device_available())


def kernel_launches():
    return int(lib().dvbt2ll_kernel_launches())


def device_count():
    return int(lib().dvbt2ll_device_count())


def set_device(device):
    if lib().dvbt2ll_set_device(int(device)) < 0:
        raise RuntimeError(last_error())


def stream_create():
    """A non-blocking stream on the current device (raw handle)."""
    s = lib().dvbt2ll_stream_create()
    if not s:
        raise RuntimeError(last_error())
    return s


def stream_destroy(s):
    lib().dvbt2ll_stream_destroy(s)


def device_synchronize():
    if lib().dvbt2ll_device_synchronize() < 0:
        raise RuntimeError(last_error())


def copy_to_host(dst, d_ptr):
    """Fill the numpy array `dst` from device memory at raw pointer d_ptr (synchronous)."""
    if lib().dvbt2ll_copy_to_host(dst.ctypes.data, d_ptr, dst.nbytes) < 0:
        raise RuntimeError(last_error())
    return dst


class DeviceBuffer(object):
    """A plain device allocation on the current device (tests and hosts without their own CUDA binding)."""

    def __init__(self, nbytes, data=None):
        self.nbytes = int(nbytes)
        self.ptr = lib().dvbt2ll_device_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError(last_error())
        if data is not None:
            data = np.ascontiguousarray(data)
            if lib().dvbt2ll_copy_to_device(self.ptr, data.ctypes.data, data.nbytes) < 0:
                raise RuntimeError(last_error())

    def to_host(self, dtype, count=None):
        out = np.empty(self.nbytes // np.dtype(dtype).itemsize if count is None else count, dtype=dtype)
        return copy_to_host(out, self.ptr)

    def free(self):
        p, self.ptr = self.ptr, None
        if p:
            lib().dvbt2ll_device_free(p)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _Block(object):
    in_dtype = np.uint8
    out_dtype = np.uint8

    def __init__(self, handle, what):
        if not handle:
            raise ValueError("%s: %s" % (what, last_error()))
        self._h = C.c_void_p(handle)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                lib().dvbt2ll_destroy(h)
            except Exception:
                pass

    @property
    def output_multiple(self):
        return lib().dvbt2ll_output_multiple(self._h)

    def forecast(self, noutput):
        return lib().dvbt2ll_forecast(self._h, noutput)

    @property
    def warnings(self):
        return lib().dvbt2ll_warnings(self._h)

    def work(self, data, nframes):
        """general_work() on host buffers for nframes frames of output. Returns (out, consumed)."""
        data = np.ascontiguousarray(data, dtype=self.in_dtype)
        nout = nframes * self.output_multiple
        out = np.empty(nout, dtype=self.out_dtype)
        consumed = C.c_int(0)
        r = lib().dvbt2ll_work(self._h, data.ctypes.data, data.size, out.ctypes.data, nout, C.byref(consumed))
        if r < 0:
            raise RuntimeError("dvbt2ll_work failed (%d): %s" % (r, last_error()))
        return out[:r], consumed.value

    def work_into(self, data, out, nframes):
        """general_work() into a caller-owned output array (long-lived buffers, as the scheduler's are).
        Returns (items produced, consumed)."""
        nout = nframes * self.output_multiple
        consumed = C.c_int(0)
        r = lib().dvbt2ll_work(self._h, data.ctypes.data, data.size, out.ctypes.data, nout, C.byref(consumed))
        if r < 0:
            raise RuntimeError("dvbt2ll_work failed (%d): %s" % (r, last_error()))
        return r, consumed.value

    def work_device(self, d_in, n_in, d_out, n_out, stream=None):
        """general_work() on DEVICE buffers (raw pointers, item counts), asynchronous on `stream` (a raw cudaStream_t;
        None = the handle's own stream followed by a synchronize). Returns (items produced, consumed)."""
        consumed = C.c_int(0)
        r = lib().dvbt2ll_work_device(self._h, C.c_void_p(d_in), int(n_in), C.c_void_p(d_out), int(n_out), C.byref(consumed),
                                      C.c_void_p(stream) if stream else None)
        if r < 0:
            raise RuntimeError("dvbt2ll_work_device failed (%d): %s" % (r, last_error()))
        return r, consumed.value

    def set_host_register(self, on=True):
        """Register the host buffers handed to work() with CUDA on first sight (only for long-lived buffers)."""
        lib().dvbt2ll_set_host_register(self._h, 1 if on else 0)

    def link_to(self, consumer, lazy_host=False):
        """Device-resident hand-off: `consumer` takes its input from HBM when it is handed what this block last wrote.
        lazy_host: this block's host output is only written when the consumer did not take the items from HBM
        (for edges whose only reader is `consumer`)."""
        r = lib().dvbt2ll_link(self._h, consumer._h)
        if r >= 0 and lazy_host:
            r = lib().dvbt2ll_link_lazy_host(self._h, 1)
        if r < 0:
            raise ValueError(last_error())

    @property
    def link_late_writes(self):
        return int(lib().dvbt2ll_link_late_writes(self._h))

    @property
    def link_hits(self):
        return int(lib().dvbt2ll_link_hits(self._h))

    def plan(self, name, dtype):
        """Host-side plan table by name (see dvbt2ll_plan_get)."""
        n = lib().dvbt2ll_plan_get(self._h, name.encode(), None, 0)
        if n < 0:
            raise KeyError(name)
        buf = np.empty(n, dtype=np.uint8)
        lib().dvbt2ll_plan_get(self._h, name.encode(), buf.ctypes.data, n)
        return buf.view(dtype)


class bbheaderbch_bb(_Block):
    """TS bytes -> BB header + scrambled BBFRAME + BCH parity, one bit per output byte."""

    def __init__(self, framesize, rate, mode, inband, fecblocks, tsrate):
        _Block.__init__(self, lib().dvbt2ll_bbheaderbch_create(framesize, rate, mode, inband, fecblocks, tsrate),
                        "bbheaderbch_bb")


class ldpc_bb(_Block):
    """The LDPC stage the shipped flowgraph places after bbheaderbch_bb (dtv.dvb_ldpc_bb, DVB-T2 codes)."""

    def __init__(self, framesize, rate):
        _Block.__init__(self, lib().dvbt2ll_ldpc_create(framesize, rate), "ldpc_bb")


class interleavermod_bc(_Block):
    out_dtype = np.complex64

    def __init__(self, framesize, rate, constellation, rotation):
        _Block.__init__(self, lib().dvbt2ll_interleavermod_create(framesize, rate, constellation, rotation),
                        "interleavermod_bc")


class framemapperfint_cc(_Block):
    in_dtype = np.complex64
    out_dtype = np.complex64

    def __init__(self, framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize,
                 guardinterval, l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble,
                 inputmode, reservedbiasbits, l1scrambled, inband):
        _Block.__init__(self, lib().dvbt2ll_framemapperfint_create(
            framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize, guardinterval,
            l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble, inputmode,
            reservedbiasbits, l1scrambled, inband), "framemapperfint_cc")


class pilotgenp1insert_cc(_Block):
    in_dtype = np.complex64
    out_dtype = np.complex64

    def __init__(self, carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble,
                 misogroup, equalization, bandwidth, vlength):
        _Block.__init__(self, lib().dvbt2ll_pilotgenp1insert_create(
            carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble, misogroup,
            equalization, bandwidth, vlength), "pilotgenp1insert_cc")


def blocks_for(cfg):
    """The five stages of the shipped flowgraph for a config dict (configs.resolve)."""
    cfg = configs.resolve(cfg)
    return dict(
        bb=bbheaderbch_bb(cfg["framesize"], cfg["rate"], cfg["inputmode"], cfg["inband"], cfg["fecblocks"], cfg["tsrate"]),
        ldpc=ldpc_bb(cfg["framesize"], cfg["rate"]),
        im=interleavermod_bc(cfg["framesize"], cfg["rate"], cfg["constellation"], cfg["rotation"]),
        fm=framemapperfint_cc(cfg["framesize"], cfg["rate"], cfg["constellation"], cfg["rotation"], cfg["fecblocks"],
                              cfg["tiblocks"], cfg["carriermode"], cfg["fftsize"], cfg["guardinterval"],
                              cfg["l1constellation"], cfg["pilotpattern"], cfg["t2frames"], cfg["numdatasyms"],
                              cfg["paprmode"], cfg["version"], cfg["preamble"], cfg["inputmode"],
                              cfg["reservedbiasbits"], cfg["l1scrambled"], cfg["inband"]),
        pg=pilotgenp1insert_cc(cfg["carriermode"], cfg["fftsize"], cfg["pilotpattern"], cfg["guardinterval"],
                               cfg["numdatasyms"], cfg["paprmode"], cfg["version"], cfg["preamble"], cfg["misogroup"],
                               cfg["equalization"], cfg["bandwidth"], cfg["vlength"]))


class Chain(_Block):
    """Fused device-resident chain: TS bytes -> complex baseband, batching channels x T2 frames."""
    out_dtype = np.complex64

    def __init__(self, cfg, max_frames, device=-1):
        cfg = configs.resolve(cfg)
        self.cfg = cfg
        p = ChainParams(**{n: int(cfg[n]) for n, _ in ChainParams._fields_})
        plps = cfg.get("plp_fecblocks")
        if cfg.get("plps"):                 # PLPs with their own FEC type, code rate, constellation and rotation
            pp = plp_params(cfg)
            arr = (PlpParams * len(pp))(*[PlpParams(**q) for q in pp])
            h = lib().dvbt2ll_chain_create_plps(C.byref(p), len(pp), arr, int(max_frames), int(device))
        elif plps and len(plps) > 1:        # several PLPs of the same parameters (beyond the single-PLP reference)
            arr = (C.c_int * len(plps))(*[int(x) for x in plps])
            h = lib().dvbt2ll_chain_create_multiplp(C.byref(p), len(plps), arr, int(max_frames), int(device))
        else:
            h = lib().dvbt2ll_chain_create(C.byref(p), int(max_frames), int(device))
        _Block.__init__(self, h, "chain")
        self.max_frames = max_frames

    @property
    def num_plp(self):
        return int(lib().dvbt2ll_chain_num_plp(self._h))

    def plp_ts_bytes(self, plp, first_frame, n_frames):
        """TS bytes PLP `plp` of one channel consumes for T2 frames [first_frame, first_frame + n_frames)."""
        return int(lib().dvbt2ll_chain_plp_ts_bytes(self._h, int(plp), int(first_frame), int(n_frames)))

    @property
    def ts_bytes_per_frame(self):
        return int(lib().dvbt2ll_chain_ts_bytes_per_frame(self._h))

    def ts_bytes(self, first_frame, n_frames):
        """TS bytes per channel consumed by T2 frames [first_frame, first_frame + n_frames)."""
        return int(lib().dvbt2ll_chain_ts_bytes(self._h, int(first_frame), int(n_frames)))

    @property
    def samples_per_frame(self):
        return int(lib().dvbt2ll_chain_samples_per_frame(self._h))

    @property
    def fecframes_per_frame(self):
        return int(lib().dvbt2ll_chain_fecframes_per_frame(self._h))

    sink_format = 0

    def set_sink(self, fmt, gain=1.0):
        """fmt 0: complex64 (default); fmt 1: interleaved int16 I/Q = round(gain * x * 32767). gain = the flowgraph's multiply_const."""
        r = lib().dvbt2ll_chain_set_sink(self._h, int(fmt), float(gain))
        if r < 0:
            raise ValueError(last_error())
        self.sink_format = int(fmt)

    def set_papr_tr(self, iterations, vclip, tone_max):
        """Tone-reservation PAPR reduction on the reserved carriers (paprmode TR or BOTH): up to `iterations` (1..64)
        peak cancellations per OFDM symbol down to the sample magnitude `vclip` (units of the complex64 output at gain
        1), no reserved carrier above `tone_max` (data cells have unit mean power); iterations = 0 switches it off.
        The "papr" tap then holds updates applied | stop reason << 8 per (channel, frame, symbol)."""
        r = lib().dvbt2ll_chain_set_papr_tr(self._h, int(iterations), float(vclip), float(tone_max))
        if r < 0:
            raise ValueError(last_error())

    def set_miso(self, on):
        """MISO processing (EN 302 755 9.1, modified Alamouti; preamble T2_MISO or T2_LITE_MISO): with on = 1 a chain
        with misogroup TX2 emits group 2, whose cells of each OFDM symbol are the pairs (-conj(g_2i+1), conj(g_2i)) of
        group 1's; with misogroup TX1 the output is unchanged.  Off by default."""
        r = lib().dvbt2ll_chain_set_miso(self._h, int(on))
        if r < 0:
            raise ValueError(last_error())

    def history_bytes(self, first_frame):
        """Stream bytes that must precede the first TS byte of `first_frame` in every row handed to run_host():
        187 in normal input mode once the stream has started (CRC-8 of the packet in flight), else 0."""
        return 187 if (first_frame > 0 and self.cfg["inputmode"] == configs.INPUTMODE_NORMAL) else 0

    def run_host(self, ts, n_channels, n_frames, first_frame=0, out=None):
        """ts: uint8 array [n_channels, history_bytes(first_frame) + >= ts_bytes(first_frame, n_frames)] (host): each row
        starts with the history bytes (the 187 stream bytes before the first frame; none for first_frame = 0 or in
        high-efficiency mode), followed by the TS bytes of the frames.  Returns complex64 [n_channels, n_frames*samples]
        (int16 [n_channels, n_frames*samples, 2] with sink format 1)."""
        ts, hist = self._host_ts(ts, n_channels, n_frames, first_frame)
        if out is None:
            out = self._host_out(n_channels, n_frames)
        r = lib().dvbt2ll_chain_run_host(self._h, ts.ctypes.data + hist, ts.shape[1], n_channels, n_frames, first_frame,
                                         out.ctypes.data)
        if r < 0:
            raise RuntimeError("dvbt2ll_chain_run_host failed (%d): %s" % (r, last_error()))
        return out

    def run_host_miso(self, ts, n_channels, n_frames, first_frame=0):
        """Both MISO transmitter groups from one pass of BB/BCH, LDPC and mapper (preamble T2_MISO or T2_LITE_MISO, tone
        reservation off): returns (out1, out2), group 1 and group 2 with MISO processing, each laid out as run_host's
        output.  ts as for run_host; misogroup does not matter."""
        ts, hist = self._host_ts(ts, n_channels, n_frames, first_frame)
        out1, out2 = self._host_out(n_channels, n_frames), self._host_out(n_channels, n_frames)
        r = lib().dvbt2ll_chain_run_host_miso(self._h, ts.ctypes.data + hist, ts.shape[1], n_channels, n_frames,
                                              first_frame, out1.ctypes.data, out2.ctypes.data)
        if r < 0:
            raise RuntimeError("dvbt2ll_chain_run_host_miso failed (%d): %s" % (r, last_error()))
        return out1, out2

    def _host_ts(self, ts, n_channels, n_frames, first_frame):
        P = self.num_plp
        ts = np.ascontiguousarray(ts, dtype=np.uint8).reshape(n_channels * P, -1)      # row = channel * num_plp + plp
        hist = self.history_bytes(first_frame)
        need = max(self.plp_ts_bytes(p, first_frame, n_frames) for p in range(P))
        if ts.shape[1] < hist + need:
            raise ValueError("run_host: each TS row needs %d history bytes + %d TS bytes, got %d" % (hist, need, ts.shape[1]))
        return ts, hist

    def _host_out(self, n_channels, n_frames):
        if self.sink_format:
            return np.empty((n_channels, n_frames * self.samples_per_frame, 2), dtype=np.int16)
        return np.empty((n_channels, n_frames * self.samples_per_frame), dtype=np.complex64)

    def run_device(self, d_ts_ptr, ts_pitch, n_channels, n_frames, first_frame, d_out_ptr, stream_ptr):
        r = lib().dvbt2ll_chain_run_device(self._h, d_ts_ptr, ts_pitch, n_channels, n_frames, first_frame, d_out_ptr,
                                           stream_ptr)
        if r < 0:
            raise RuntimeError("dvbt2ll_chain_run_device failed (%d): %s" % (r, last_error()))
        return r

    def run_device_miso(self, d_ts_ptr, ts_pitch, n_channels, n_frames, first_frame, d_out1_ptr, d_out2_ptr, stream_ptr):
        """run_device with both MISO groups from one front-end pass: group 1 to d_out1_ptr, group 2 with MISO processing
        to d_out2_ptr (see run_host_miso)."""
        r = lib().dvbt2ll_chain_run_device_miso(self._h, d_ts_ptr, ts_pitch, n_channels, n_frames, first_frame,
                                                d_out1_ptr, d_out2_ptr, stream_ptr)
        if r < 0:
            raise RuntimeError("dvbt2ll_chain_run_device_miso failed (%d): %s" % (r, last_error()))
        return r

    def tap(self, stage, dtype=np.uint8):
        """Stage output of the most recent run: "bch", "fec", "cells", one PLP's codewords "bch.<p>" / "fec.<p>", or the
        tone-reservation counts "papr" (int16)."""
        n = lib().dvbt2ll_chain_tap(self._h, stage.encode(), None, 0)
        if n < 0:
            raise RuntimeError(last_error())
        buf = np.empty(n, dtype=np.uint8)
        lib().dvbt2ll_chain_tap(self._h, stage.encode(), buf.ctypes.data, n)
        return buf.view(dtype)

    def enable_timing(self, on=True):
        lib().dvbt2ll_chain_enable_timing(self._h, 1 if on else 0)

    def stage_ms(self):
        ms = (C.c_float * 5)()
        r = lib().dvbt2ll_chain_stage_ms(self._h, ms)
        if r < 0:
            raise RuntimeError(last_error())
        return dict(zip(("bb_bch", "ldpc", "map", "ofdm", "total"), [float(x) for x in ms]))


def ts_sync(ts):
    """First offset at which 0x47 repeats every 188 bytes over 5 packets (-1: none)."""
    ts = np.ascontiguousarray(ts, dtype=np.uint8)
    return int(lib().dvbt2ll_ts_sync(ts.ctypes.data, ts.size))


def ts_fill(src, pos, nbytes):
    """Bytes [pos, pos + nbytes) of the packet-aligned stream `src`, continued with null packets past its last whole
    packet (zeros for pos < 0). Returns (bytes, null-packet bytes inserted)."""
    src = np.ascontiguousarray(src, dtype=np.uint8)
    out = np.empty(nbytes, dtype=np.uint8)
    n = lib().dvbt2ll_ts_fill(out.ctypes.data, nbytes, src.ctypes.data, src.size, int(pos))
    return out, int(n)


def set_auto_link(on=True):
    """Process-wide: drop-in blocks keep their outputs resident and find their input among the other blocks' resident
    outputs by host address -- the device-resident hand-off without link_to() (dvbt2ll_set_auto_link)."""
    lib().dvbt2ll_set_auto_link(1 if on else 0)


def set_overfull_policy(warn):
    """False (default): creating a frame mapper / chain whose T2 frame is over-full fails; True: warn and truncate
    like the reference (lib/framemapperfint_cc_impl.cc:1138-1141)."""
    lib().dvbt2ll_set_overfull_policy(1 if warn else 0)


class Gather(object):
    """Ordered multi-GPU reassembly on the root GPU (dvbt2ll_gather_*): see include/dvbt2ll_cuda.h.
    `exchange(blob_bytes) -> list of every rank's blob in rank order` is the only host-side collective (done once);
    bench.py passes a torch.distributed all_gather."""

    def __init__(self, rank, world, root, device, slot_bytes, local_bytes, n_slots=2):
        self.rank, self.world, self.root = rank, world, root
        h = lib().dvbt2ll_gather_create(rank, world, root, device, slot_bytes, local_bytes, n_slots)
        if not h:
            raise RuntimeError("dvbt2ll_gather_create: %s" % lib().dvbt2ll_gather_last_error().decode())
        self._h = C.c_void_p(h)

    def _ck(self, r, what):
        if r < 0:
            raise RuntimeError("%s failed (%d): %s" % (what, r, lib().dvbt2ll_gather_last_error().decode()))
        return r

    def export(self):
        buf = (C.c_ubyte * GATHER_BLOB_BYTES)()
        self._ck(lib().dvbt2ll_gather_export(self._h, buf, GATHER_BLOB_BYTES), "gather_export")
        return bytes(buf)

    def connect(self, blobs):
        raw = b"".join(blobs)
        self._ck(lib().dvbt2ll_gather_connect(self._h, raw, len(raw)), "gather_connect")

    def acquire(self, step, offset, producer_stream):
        p = C.c_void_p(0)
        self._ck(lib().dvbt2ll_gather_acquire(self._h, step, offset, producer_stream, C.byref(p)), "gather_acquire")
        return p.value

    def push(self, step, offset, nbytes, producer_stream):
        self._ck(lib().dvbt2ll_gather_push(self._h, step, offset, nbytes, producer_stream), "gather_push")

    def wait(self, step, consumer_stream):
        p = C.c_void_p(0)
        self._ck(lib().dvbt2ll_gather_wait(self._h, step, consumer_stream, C.byref(p)), "gather_wait")
        return p.value

    def release(self, step, consumer_stream):
        self._ck(lib().dvbt2ll_gather_release(self._h, step, consumer_stream), "gather_release")

    @property
    def side_stream(self):
        return lib().dvbt2ll_gather_side_stream(self._h)

    def close(self):
        h, self._h = self._h, None
        if h:
            lib().dvbt2ll_gather_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
