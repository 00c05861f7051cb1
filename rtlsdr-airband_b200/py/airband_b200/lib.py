"""ctypes binding of the product: rtlsdr-airband_b200/libairband_b200.so (C ABI in include/airband_b200.h).

There is no fallback of any kind here: if the shared library is missing, or no sm_100 device is present,
construction raises.  (The CPU oracle under oracle/ is test infrastructure and is never imported from here.)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .config import CConfig, CSquelchStats, Config

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.abspath(os.path.join(_HERE, "..", ".."))
LIB_PATH = os.environ.get("ABG_LIB_PATH") or os.path.join(LIB_DIR, "libairband_b200.so")  # override: A/B-testing builds

# every symbol include/airband_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "abg_last_error", "abg_version", "abg_create", "abg_destroy", "abg_wave_batch", "abg_hop", "abg_push",
    "abg_batches_available", "abg_run", "abg_sync", "abg_join", "abg_batches_ready", "abg_fetch_batch", "abg_fetch_batches", "abg_get_stats", "abg_set_bin",
    "abg_resident_load", "abg_run_resident", "abg_set_stream", "abg_launch_count", "abg_mixers_configure",
    "abg_fetch_mixer_batch", "abg_mixer_device_buffers", "abg_debug_frame", "abg_last_run_times", "abg_debug_timeline", "abg_scan_configure", "abg_scan_select", "abg_host_register", "abg_host_unregister", "abg_ingest_sync", "abg_fft_path", "abg_debug_tc_table", "abg_debug_inject_wavein", "abg_debug_k1tc_trace", "abg_debug_k2_stats",
    "abg_push_device", "abg_ingest_join", "abg_set_result_location", "abg_fetch_batches_device", "abg_fetch_all_device",
    "abg_fetch_mixer_batches_device",
]

RESULTS_HOST, RESULTS_DEVICE = 0, 1  # abg_set_result_location


class COptions(C.Structure):
    _fields_ = [
        ("cuda_device", C.c_int32),
        ("max_batches_per_run", C.c_int32),
        ("input_capacity_batches", C.c_int32),
        ("fft_mode", C.c_int32),
        ("reserved", C.c_int32 * 4),
    ]


class CMixerInput(C.Structure):
    _fields_ = [("dev", C.c_int32), ("chan", C.c_int32), ("ampfactor", C.c_float), ("balance", C.c_float)]


class AbgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"airband_b200 error {code}: {msg}")
        self.code = code


_LIB = None


def load():
    """dlopen the engine library (raises FileNotFoundError with build instructions if it has not been built)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                f"(or `make -C {LIB_DIR}`) first. There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i, f = C.c_void_p, C.c_int, C.c_float
    L.abg_last_error.restype, L.abg_last_error.argtypes = C.c_char_p, []
    L.abg_version.restype, L.abg_version.argtypes = C.c_char_p, []
    L.abg_create.restype, L.abg_create.argtypes = i, [C.POINTER(CConfig), C.POINTER(COptions), C.POINTER(vp)]
    L.abg_destroy.restype, L.abg_destroy.argtypes = None, [vp]
    L.abg_wave_batch.restype, L.abg_wave_batch.argtypes = i, [vp]
    L.abg_hop.restype, L.abg_hop.argtypes = i, [vp, i]
    L.abg_push.restype, L.abg_push.argtypes = i, [vp, i, vp, C.c_size_t]
    L.abg_batches_available.restype, L.abg_batches_available.argtypes = i, [vp, i]
    L.abg_run.restype, L.abg_run.argtypes = i, [vp, i]
    L.abg_sync.restype, L.abg_sync.argtypes = i, [vp]
    L.abg_join.restype, L.abg_join.argtypes = i, [vp]
    L.abg_batches_ready.restype, L.abg_batches_ready.argtypes = i, [vp, i]
    L.abg_fetch_batch.restype, L.abg_fetch_batch.argtypes = i, [vp, i, vp, vp, vp]
    L.abg_fetch_batches.restype, L.abg_fetch_batches.argtypes = i, [vp, i, i, vp, vp, vp]
    L.abg_get_stats.restype, L.abg_get_stats.argtypes = i, [vp, i, i, C.POINTER(CSquelchStats)]
    L.abg_set_bin.restype, L.abg_set_bin.argtypes = i, [vp, i, i, i]
    L.abg_resident_load.restype, L.abg_resident_load.argtypes = i, [vp, i, vp, C.c_size_t]
    L.abg_run_resident.restype, L.abg_run_resident.argtypes = i, [vp, i]
    L.abg_set_stream.restype, L.abg_set_stream.argtypes = i, [vp, vp]
    L.abg_launch_count.restype, L.abg_launch_count.argtypes = C.c_uint64, [vp]
    L.abg_mixers_configure.restype, L.abg_mixers_configure.argtypes = i, [vp, i, C.POINTER(C.c_int32), C.POINTER(CMixerInput)]
    L.abg_fetch_mixer_batch.restype, L.abg_fetch_mixer_batch.argtypes = i, [vp, i, vp, vp, C.POINTER(C.c_int)]
    L.abg_mixer_device_buffers.restype, L.abg_mixer_device_buffers.argtypes = i, [vp, C.POINTER(vp), C.POINTER(vp)]
    L.abg_debug_frame.restype, L.abg_debug_frame.argtypes = i, [vp, i, vp, vp]
    L.abg_last_run_times.restype, L.abg_last_run_times.argtypes = i, [vp, C.POINTER(C.c_float)]
    L.abg_host_register.restype, L.abg_host_register.argtypes = i, [vp, C.c_size_t]
    L.abg_host_unregister.restype, L.abg_host_unregister.argtypes = i, [vp]
    L.abg_ingest_sync.restype, L.abg_ingest_sync.argtypes = i, [vp]
    L.abg_scan_configure.restype, L.abg_scan_configure.argtypes = i, [vp, i, i, i, vp]
    L.abg_scan_select.restype, L.abg_scan_select.argtypes = i, [vp, i, i, i]
    L.abg_debug_timeline.restype, L.abg_debug_timeline.argtypes = i, [vp, i, C.POINTER(C.c_float)]
    L.abg_fft_path.restype, L.abg_fft_path.argtypes = i, [vp, i]
    L.abg_debug_inject_wavein.restype, L.abg_debug_inject_wavein.argtypes = i, [vp, i, i, vp]
    L.abg_debug_k1tc_trace.restype, L.abg_debug_k1tc_trace.argtypes = i, [vp]
    L.abg_debug_k2_stats.restype, L.abg_debug_k2_stats.argtypes = i, [vp]
    L.abg_push_device.restype, L.abg_push_device.argtypes = i, [vp, i, vp, C.c_size_t, vp]
    L.abg_ingest_join.restype, L.abg_ingest_join.argtypes = i, [vp, vp]
    L.abg_set_result_location.restype, L.abg_set_result_location.argtypes = i, [vp, i]
    L.abg_fetch_batches_device.restype, L.abg_fetch_batches_device.argtypes = i, [vp, i, i, vp, vp, vp, vp]
    L.abg_fetch_all_device.restype, L.abg_fetch_all_device.argtypes = i, [vp, i, vp, vp, vp, vp]
    L.abg_fetch_mixer_batches_device.restype, L.abg_fetch_mixer_batches_device.argtypes = i, [vp, i, vp, vp, vp]
    L.abg_debug_tc_table.restype = i
    L.abg_debug_tc_table.argtypes = [i, i, i, f, i, vp, i, vp, vp, C.c_size_t, vp, C.POINTER(C.c_double)]
    _LIB = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Engine:
    """One engine = one GPU's contiguous range of devices[] (a demod_params_t{device_start, device_end})."""

    def __init__(self, cfg: Config, *, cuda_device: int = -1, max_batches_per_run: int = 4, input_capacity_batches: int = 0,
                 fft_mode: int = 0):
        self.L = load()
        self.cfg = cfg
        ccfg, self._keep = cfg.to_c()
        opt = COptions(cuda_device, max_batches_per_run, input_capacity_batches, fft_mode)
        h = C.c_void_p()
        self.h = None
        self._chk(self.L.abg_create(C.byref(ccfg), C.byref(opt), C.byref(h)))
        self.h = h
        self.B = self.L.abg_wave_batch(self.h)
        self.nbmax = max_batches_per_run
        self.cuda_device = cuda_device  # -1: the CUDA device that was current at creation
        self.G = sum(len(d.channels) for d in cfg.devices)
        self._n_mixers = 0

    def _chk(self, rc: int) -> int:
        if rc < 0:
            raise AbgError(rc, (self.L.abg_last_error() or b"").decode())
        return rc

    def close(self):
        if self.h:
            self.L.abg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- streaming path -------------------------------------------------------------------------------------------
    def push(self, dev: int, raw: np.ndarray) -> None:
        raw = np.ascontiguousarray(raw)
        self._chk(self.L.abg_push(self.h, dev, _ptr(raw), raw.nbytes))

    def push_ptr(self, dev: int, ptr: int, nbytes: int) -> None:
        self._chk(self.L.abg_push(self.h, dev, C.c_void_p(ptr), nbytes))

    def batches_available(self, dev: int) -> int:
        return self._chk(self.L.abg_batches_available(self.h, dev))

    def run(self, max_batches: int = -1) -> int:
        return self._chk(self.L.abg_run(self.h, max_batches))

    def sync(self) -> None:
        self._chk(self.L.abg_sync(self.h))

    def join(self) -> None:
        self._chk(self.L.abg_join(self.h))

    def batches_ready(self, dev: int) -> int:
        return self._chk(self.L.abg_batches_ready(self.h, dev))

    def fetch(self, dev: int, want_iq: bool = True) -> Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        Cn = len(self.cfg.devices[dev].channels)
        wo = np.empty((Cn, self.B), np.float32)
        iq = np.empty((Cn, 2 * self.B), np.float32) if want_iq else None
        ax = np.empty(Cn, np.uint8)
        if not self._chk(self.L.abg_fetch_batch(self.h, dev, _ptr(wo), _ptr(iq), _ptr(ax))):
            return None
        return wo, (iq.view(np.complex64) if iq is not None else None), ax

    def fetch_into(self, dev: int, wo: np.ndarray, ax: np.ndarray) -> bool:
        return bool(self._chk(self.L.abg_fetch_batch(self.h, dev, _ptr(wo), None, _ptr(ax))))

    def fetch_many_into(self, dev: int, max_batches: int, wo: np.ndarray, ax: np.ndarray) -> int:
        """Pop up to max_batches batches of a device into wo[n, C, B] / ax[n, C]; returns how many."""
        return self._chk(self.L.abg_fetch_batches(self.h, dev, max_batches, _ptr(wo), None, _ptr(ax)))

    def fetch_all(self, dev: int):
        wos, iqs, axs = [], [], []
        while True:
            r = self.fetch(dev)
            if r is None:
                break
            wos.append(r[0]); iqs.append(r[1]); axs.append(r[2])
        Cn = len(self.cfg.devices[dev].channels)
        if not wos:
            return np.zeros((Cn, 0), np.float32), np.zeros((Cn, 0), np.complex64), np.zeros((0, Cn), np.uint8)
        return np.concatenate(wos, 1), np.concatenate(iqs, 1), np.stack(axs, 0)

    def stats(self, dev: int, chan: int) -> CSquelchStats:
        s = CSquelchStats()
        self._chk(self.L.abg_get_stats(self.h, dev, chan, C.byref(s)))
        return s

    def fft_path(self, dev: int) -> int:
        """1 full-spectrum FFT, 2 output-pruned FFT, 3 tensor-core DFT (which K1 the device's frames go through)."""
        return self._chk(self.L.abg_fft_path(self.h, dev))

    def set_bin(self, dev: int, chan: int, bin_: int) -> None:
        self._chk(self.L.abg_set_bin(self.h, dev, chan, bin_))

    # ---- GPU-resident I/O (torch CUDA tensors; torch is imported only here) ------------------------------------------
    # Every method runs on torch.cuda.current_stream() of the engine's GPU and never waits on the host.
    def results_on_device(self) -> None:
        """Keep result slots in HBM (ABG_RESULTS_DEVICE); needed by the fetch_*_tensors methods.  Before the first run."""
        self._chk(self.L.abg_set_result_location(self.h, RESULTS_DEVICE))

    def _torch_device(self):
        import torch
        return torch.device("cuda", self.cuda_device if self.cuda_device >= 0 else torch.cuda.current_device())

    def _stream(self) -> int:
        import torch
        return torch.cuda.current_stream(self._torch_device()).cuda_stream

    def push_device_ptr(self, dev: int, ptr: int, nbytes: int, stream: Optional[int] = None) -> None:
        """abg_push_device on raw device memory, ordered after the work enqueued so far on `stream` (default: current)."""
        self._chk(self.L.abg_push_device(self.h, dev, C.c_void_p(ptr), nbytes, C.c_void_p(self._stream() if stream is None else stream)))

    def ingest_join(self, stream: Optional[int] = None) -> None:
        self._chk(self.L.abg_ingest_join(self.h, C.c_void_p(self._stream() if stream is None else stream)))

    def push_tensor(self, dev: int, t) -> None:
        """Push ring-format samples from a contiguous CUDA tensor on the engine's GPU: uint8 for U8 devices, int8 for S8,
        int16 for S16, float32 or complex64 for F32.  The current stream then waits until the engine has copied the
        samples out, so the tensor may be overwritten or freed by work enqueued on that stream afterwards."""
        import torch
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"push_tensor expects a torch.Tensor, got {type(t).__name__}")
        if not 0 <= dev < len(self.cfg.devices):
            raise ValueError(f"device {dev} out of range")
        from .config import SFMT_U8, SFMT_S8, SFMT_S16, SFMT_F32
        want = {SFMT_U8: (torch.uint8,), SFMT_S8: (torch.int8,), SFMT_S16: (torch.int16,),
                SFMT_F32: (torch.float32, torch.complex64)}[self.cfg.devices[dev].sfmt]
        if t.dtype not in want:
            raise TypeError(f"device {dev} takes {' or '.join(str(w) for w in want)} samples, got {t.dtype}")
        if not t.is_cuda:
            raise ValueError("push_tensor expects a CUDA tensor (use push() for host memory)")
        if not t.is_contiguous():
            raise ValueError("push_tensor expects a contiguous tensor")
        if self.cuda_device >= 0 and t.device.index != self.cuda_device:
            raise ValueError(f"tensor is on cuda:{t.device.index}, the engine on cuda:{self.cuda_device}")
        stream = torch.cuda.current_stream(t.device).cuda_stream
        nbytes = t.numel() * t.element_size()
        self._chk(self.L.abg_push_device(self.h, dev, C.c_void_p(t.data_ptr()), nbytes, C.c_void_p(stream)))
        self._chk(self.L.abg_ingest_join(self.h, C.c_void_p(stream)))

    def _result_tensors(self, n: int, rows: int, want_iq: bool):
        import torch
        dv = self._torch_device()
        wo = torch.empty((n, rows, self.B), dtype=torch.float32, device=dv)
        iq = torch.empty((n, rows, self.B), dtype=torch.complex64, device=dv) if want_iq else None
        ax = torch.empty((n, rows), dtype=torch.uint8, device=dv)
        return wo, iq, ax

    @staticmethod
    def _tptr(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    def fetch_tensors(self, dev: int, max_batches: int, want_iq: bool = True, out=None):
        """Pop up to max_batches finished batches of a device into CUDA tensors: (waveout float32[n, C, B],
        iq_out complex64[n, C, B] or None, axcindicate uint8[n, C]).  `out` = preallocated tensors of at least that size."""
        n = min(max_batches, self.batches_ready(dev))
        Cn = len(self.cfg.devices[dev].channels)
        wo, iq, ax = out if out is not None else self._result_tensors(n, Cn, want_iq)
        got = self._chk(self.L.abg_fetch_batches_device(self.h, dev, n, self._tptr(wo), self._tptr(iq), self._tptr(ax),
                                                        C.c_void_p(self._stream())))
        return wo[:got], (iq[:got] if iq is not None else None), ax[:got]

    def fetch_all_tensors(self, n_batches: int, want_iq: bool = True, out=None):
        """Pop n_batches batches of every device in one launch: (waveout float32[n, G, B], iq_out complex64[n, G, B] or
        None, axcindicate uint8[n, G]), G = every channel of the engine in device order."""
        wo, iq, ax = out if out is not None else self._result_tensors(n_batches, self.G, want_iq)
        got = self._chk(self.L.abg_fetch_all_device(self.h, n_batches, self._tptr(wo), self._tptr(iq), self._tptr(ax),
                                                    C.c_void_p(self._stream())))
        return wo[:got], (iq[:got] if iq is not None else None), ax[:got]

    def fetch_mixer_tensors(self, max_batches: int):
        """Pop up to max_batches batches of every mixer: (left_right float32[n, n_mixers, 2, B], has_signal int32[n, n_mixers])."""
        import torch
        M, dv = self._n_mixers, self._torch_device()
        lr = torch.empty((max_batches, M, 2, self.B), dtype=torch.float32, device=dv)
        hs = torch.empty((max_batches, M), dtype=torch.int32, device=dv)
        got = self._chk(self.L.abg_fetch_mixer_batches_device(self.h, max_batches, self._tptr(lr), self._tptr(hs), C.c_void_p(self._stream())))
        return lr[:got], hs[:got]

    # ---- resident (benchmark) path -------------------------------------------------------------------------------
    def resident_load(self, dev: int, raw: np.ndarray) -> None:
        raw = np.ascontiguousarray(raw)
        self._chk(self.L.abg_resident_load(self.h, dev, _ptr(raw), raw.nbytes))

    def resident_bytes_needed(self, dev: int) -> int:
        d = self.cfg.devices[dev]
        hop_b = self.cfg.hop(dev) * 2 * d.bytes_per_sample
        return (self.nbmax * self.B + 100 - 1) * hop_b + self.cfg.fft_size * 2 * d.bytes_per_sample

    def run_resident(self, n_batches: int) -> int:
        return self._chk(self.L.abg_run_resident(self.h, n_batches))

    def set_stream(self, cuda_stream_ptr: int) -> None:
        self._chk(self.L.abg_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def last_run_times(self):
        """(k1_ms, k2_ms, tail_ms, total_ms) of the most recent run, from CUDA events on the engine's stream."""
        a = (C.c_float * 4)()
        self._chk(self.L.abg_last_run_times(self.h, a))
        return tuple(float(x) for x in a)

    def timeline(self, n_runs: int = 8) -> np.ndarray:
        """[n_runs, 5] ms: K1 start, K1 end, K2 start, K2 end, end of run, relative to the oldest run's K1 start."""
        a = (C.c_float * (5 * n_runs))()
        self._chk(self.L.abg_debug_timeline(self.h, n_runs, a))
        return np.array(a, dtype=np.float32).reshape(n_runs, 5)

    def scan_configure(self, dev: int, chan: int, freqs) -> None:
        """Install a scan-mode frequency list (list of config.Channel); entry 0 becomes current."""
        from .config import channels_to_c
        arr = channels_to_c(freqs)
        self._chk(self.L.abg_scan_configure(self.h, dev, chan, len(freqs), C.cast(arr, C.c_void_p)))

    def scan_select(self, dev: int, chan: int, freq_idx: int) -> None:
        self._chk(self.L.abg_scan_select(self.h, dev, chan, freq_idx))

    def launch_count(self) -> int:
        return int(self.L.abg_launch_count(self.h))

    # ---- mixers ---------------------------------------------------------------------------------------------------
    def configure_mixers(self, mixers: Sequence[Sequence[Tuple[int, int, float, float]]]) -> None:
        """mixers[m] = [(dev, chan, ampfactor, balance), ...]"""
        self._n_mixers = len(mixers)
        offs = [0]
        flat = []
        for m in mixers:
            flat.extend(m)
            offs.append(len(flat))
        arr = (CMixerInput * max(1, len(flat)))()
        for k, (d, c, a, b) in enumerate(flat):
            arr[k] = CMixerInput(d, c, a, b)
        co = (C.c_int32 * len(offs))(*offs)
        self._chk(self.L.abg_mixers_configure(self.h, len(mixers), co, arr))

    def fetch_mixer(self, mixer: int):
        left = np.empty(self.B, np.float32)
        right = np.empty(self.B, np.float32)
        sig = C.c_int(0)
        if not self._chk(self.L.abg_fetch_mixer_batch(self.h, mixer, _ptr(left), _ptr(right), C.byref(sig))):
            return None
        return left, right, bool(sig.value)

    def mixer_device_buffers(self) -> Tuple[int, int]:
        a, b = C.c_void_p(), C.c_void_p()
        self._chk(self.L.abg_mixer_device_buffers(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def inject_wavein(self, dev: int, wavein: np.ndarray) -> int:
        """Stage tap: wavein[C, n_batches * B] straight into the demodulation state machine (K1 skipped)."""
        w = np.ascontiguousarray(wavein, np.float32)
        assert w.ndim == 2 and w.shape[1] % self.B == 0
        return self._chk(self.L.abg_debug_inject_wavein(self.h, dev, w.shape[1] // self.B, _ptr(w)))

    # ---- stage tap ------------------------------------------------------------------------------------------------
    def debug_frame(self, dev: int, raw_frame: np.ndarray) -> np.ndarray:
        out = np.empty(2 * self.cfg.fft_size, np.float32)
        raw_frame = np.ascontiguousarray(raw_frame)
        self._chk(self.L.abg_debug_frame(self.h, dev, _ptr(raw_frame), _ptr(out)))
        return out.view(np.complex64)


TC_PLAN_FIELDS = ("eligible", "K", "HC", "S", "NC", "ND", "C2p", "KBS", "NSTB", "tmem_cols", "smem_bytes", "halo", "nacc")


def tc_table(fft_size: int, sfmt: int, hop_bytes: int, bins: Sequence[int], digits: int = 4, fullscale: float = 1.0):
    """Host-only view of the tensor-core K1's plan and coefficient table (abg_debug_tc_table).  Returns (plan dict,
    tab int8[K/32, 2, NC, 16], sq int64[C2p], cscale) or (plan, None, None, None) when the shape is not eligible."""
    L = load()
    plan = np.zeros(13, np.int32)
    b = np.asarray(bins, np.int32)
    L.abg_debug_tc_table(fft_size, sfmt, hop_bytes, fullscale, len(b), _ptr(b), digits, _ptr(plan), None, 0, None, None)
    pd = dict(zip(TC_PLAN_FIELDS, (int(x) for x in plan)))
    if not pd["eligible"]:
        return pd, None, None, None
    tab = np.zeros(pd["K"] * pd["NC"], np.int8)
    sq = np.zeros(pd["C2p"], np.int64)
    cs = C.c_double(0.0)
    rc = L.abg_debug_tc_table(fft_size, sfmt, hop_bytes, fullscale, len(b), _ptr(b), digits, _ptr(plan), _ptr(tab), tab.nbytes, _ptr(sq), C.byref(cs))
    if rc < 0:
        raise AbgError(rc, (L.abg_last_error() or b"").decode())
    return pd, tab.reshape(pd["K"] // 32, 2, pd["NC"], 16), sq, cs.value


def demodulate_all(cfg: Config, raws: List[np.ndarray], *, max_batches_per_run: int = 4, chunk_batches: int = 0, **kw):
    """Push one raw stream per device and run to exhaustion (the file-input use of the path).  Returns per-device
    (waveout[C, n], iq_out[C, n], axc[nb, C]) and the engine."""
    e = Engine(cfg, max_batches_per_run=max_batches_per_run, **kw)
    pos = [0] * len(raws)
    outs = [([], [], []) for _ in raws]
    step_b = chunk_batches or max_batches_per_run
    while True:
        progressed = False
        for d, r in enumerate(raws):
            if pos[d] < r.size:
                hop_items = cfg.hop(d) * 2  # array items per hop (I and Q)
                n = step_b * e.B * hop_items + (100 * hop_items + 2 * cfg.fft_size if pos[d] == 0 else 0)
                e.push(d, r[pos[d]:pos[d] + n])
                pos[d] += n
                progressed = True
        n = e.run(-1)
        for d in range(len(raws)):
            while True:
                got = e.fetch(d)
                if got is None:
                    break
                for k in range(3):
                    outs[d][k].append(got[k])
        if n == 0 and not progressed:
            break
    res = []
    for d in range(len(raws)):
        Cn = len(cfg.devices[d].channels)
        if outs[d][0]:
            res.append((np.concatenate(outs[d][0], 1), np.concatenate(outs[d][1], 1), np.stack(outs[d][2], 0)))
        else:
            res.append((np.zeros((Cn, 0), np.float32), np.zeros((Cn, 0), np.complex64), np.zeros((0, Cn), np.uint8)))
    return res, e
