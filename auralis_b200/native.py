"""ctypes binding of ``libxtts_b200.so`` (C ABI: ``include/xtts_b200.h``).

No torch types cross this boundary: numpy arrays in host memory in, numpy arrays out.
The library is CUDA-only; creating an engine without an sm_100 GPU raises ``NativeError``
(there is no CPU fallback — parity claims depend on that).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import numpy as np

from .config import XTTSDims

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxtts_b200.so")

PRECISION_FP32 = 0
PRECISION_BF16 = 1
PRECISION_FP16 = 2
ERR_CANCELLED = -5


class NativeError(RuntimeError):
    pass


class XttsConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("precision", C.c_int32), ("max_batch", C.c_int32), ("max_speakers", C.c_int32),
        ("hidden", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32), ("ff", C.c_int32),
        ("n_text_tokens", C.c_int32), ("n_audio_tokens", C.c_int32), ("start_audio_token", C.c_int32),
        ("stop_audio_token", C.c_int32), ("max_audio_tokens", C.c_int32), ("max_text_tokens", C.c_int32),
        ("n_cond_latents", C.c_int32), ("ln_eps", C.c_float),
        ("voc_in_dim", C.c_int32), ("voc_init_ch", C.c_int32), ("voc_n_up", C.c_int32),
        ("voc_up_rates", C.c_int32 * 4), ("voc_up_kernels", C.c_int32 * 4), ("voc_n_rb", C.c_int32),
        ("voc_rb_kernels", C.c_int32 * 4), ("voc_rb_dilations", C.c_int32 * 4), ("d_vector", C.c_int32),
        ("code_stride", C.c_int32), ("output_hop_length", C.c_int32), ("input_sample_rate", C.c_int32),
        ("output_sample_rate", C.c_int32),
        ("n_mels", C.c_int32), ("cond_blocks", C.c_int32), ("perceiver_depth", C.c_int32),
        ("perceiver_heads", C.c_int32), ("perceiver_dim_head", C.c_int32), ("perceiver_ff_mult", C.c_int32),
        ("spk_layers", C.c_int32 * 4), ("spk_filters", C.c_int32 * 4), ("spk_mels", C.c_int32), ("spk_proj", C.c_int32),
    ]


class XttsSampling(C.Structure):
    _fields_ = [("temperature", C.c_float), ("top_p", C.c_float), ("repetition_penalty", C.c_float),
                ("top_k", C.c_int32), ("max_tokens", C.c_int32), ("stop_token", C.c_int32),
                ("seed", C.c_uint64), ("seq_seed", C.c_int32), ("vocode", C.c_int32), ("priority", C.c_int32),
                ("early_tokens", C.c_int32)]


class XttsResult(C.Structure):
    _fields_ = [("seq_id", C.c_uint64), ("status", C.c_int32), ("n_tokens", C.c_int32), ("n_samples", C.c_int32),
                ("n_prompt_rows", C.c_int32), ("t_submit", C.c_double), ("t_first_token", C.c_double),
                ("t_done", C.c_double)]


class XttsStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("decode_steps", C.c_uint64), ("prefill_rows", C.c_uint64),
                ("tokens_generated", C.c_uint64), ("samples_generated", C.c_uint64),
                ("gpt_ms", C.c_double), ("vocoder_ms", C.c_double), ("cond_ms", C.c_double),
                ("hbm_bytes_weights", C.c_uint64)]


class XttsKernelProfile(C.Structure):
    _fields_ = [("n", C.c_int32), ("name", (C.c_char * 32) * 16), ("ms", C.c_double * 16), ("flops", C.c_double * 16),
                ("bytes", C.c_double * 16), ("launches", C.c_uint64 * 16)]


# every symbol include/xtts_b200.h declares (checked by tests/test_abi.py against the header text)
ABI_SYMBOLS = [
    "xtts_last_error", "xtts_version", "xtts_create", "xtts_destroy", "xtts_load_weight", "xtts_finalize_weights",
    "xtts_set_speaker", "xtts_get_speaker", "xtts_condition", "xtts_submit", "xtts_cancel", "xtts_poll", "xtts_fetch",
    "xtts_set_option", "xtts_get_stats", "xtts_sync", "xtts_get_kernel_profile", "xtts_device_timer", "xtts_vocode", "xtts_vocode_window", "xtts_gpt_prefill", "xtts_gpt_teacher_forced",
    "xtts_debug_gemm", "xtts_debug_sample", "xtts_debug_trace",
]

_lib = None


def load_library(path: Optional[str] = None):
    """dlopen the library and declare prototypes.  Raises NativeError if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise NativeError(f"{p} not found: run `python -m auralis_b200.build` (no CPU fallback exists)")
    lib = C.CDLL(p)
    vp, i32, i64, f32p, i32p = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_int32)
    lib.xtts_last_error.restype = C.c_char_p
    lib.xtts_version.restype = C.c_char_p
    lib.xtts_create.argtypes = [C.POINTER(XttsConfig), C.POINTER(vp)]
    lib.xtts_destroy.argtypes = [vp]
    lib.xtts_load_weight.argtypes = [vp, C.c_char_p, f32p, C.POINTER(i64), i32]
    lib.xtts_finalize_weights.argtypes = [vp]
    lib.xtts_set_speaker.argtypes = [vp, i32, f32p, f32p]
    lib.xtts_get_speaker.argtypes = [vp, i32, f32p, f32p]
    lib.xtts_condition.argtypes = [vp, i32, f32p, i64, f32p, i64, i32, i32]
    lib.xtts_submit.argtypes = [vp, C.c_uint64, i32p, i32, i32, C.POINTER(XttsSampling)]
    lib.xtts_cancel.argtypes = [vp, C.c_uint64]
    lib.xtts_poll.argtypes = [vp, C.POINTER(XttsResult), i32]
    lib.xtts_fetch.argtypes = [vp, C.c_uint64, i32p, f32p, f32p]
    lib.xtts_set_option.argtypes = [vp, C.c_char_p, i64]
    lib.xtts_get_stats.argtypes = [vp, C.POINTER(XttsStats)]
    lib.xtts_sync.argtypes = [vp]
    lib.xtts_get_kernel_profile.argtypes = [vp, C.POINTER(XttsKernelProfile)]
    lib.xtts_device_timer.argtypes = [vp, i32, C.POINTER(C.c_double)]
    lib.xtts_vocode.argtypes = [vp, f32p, i32, i32, f32p, i32p, C.c_char_p, f32p, i64]
    lib.xtts_vocode_window.argtypes = [vp, f32p, i32, i32, i32, i32, f32p]
    lib.xtts_gpt_prefill.argtypes = [vp, i32p, i32, i32, i32p, i32, f32p, f32p, f32p]
    lib.xtts_gpt_teacher_forced.argtypes = [vp, i32p, i32, i32, i32p, i32, C.POINTER(XttsSampling), f32p, f32p, i32p]
    lib.xtts_debug_gemm.argtypes = [vp, i32, f32p, f32p, f32p, f32p, f32p, i32, i32, i32, i32, i32, f32p]
    lib.xtts_debug_sample.argtypes = [vp, f32p, C.POINTER(C.c_uint8), i32, i32, C.POINTER(XttsSampling), i32, i32p]
    lib.xtts_debug_trace.argtypes = [vp, i32, C.POINTER(C.c_uint64), i32]
    for s in ABI_SYMBOLS:
        if s not in ("xtts_last_error", "xtts_version"):
            getattr(lib, s).restype = C.c_int
    _lib = lib
    return lib


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


def _fp(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def _ip(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


def make_config(dims: XTTSDims, device: int = 0, precision: int = PRECISION_FP32, max_batch: int = 64,
                max_speakers: int = 16) -> XttsConfig:
    g, v, c = dims.gpt, dims.voc, dims.cond
    cfg = XttsConfig()
    cfg.device, cfg.precision, cfg.max_batch, cfg.max_speakers = device, precision, max_batch, max_speakers
    cfg.hidden, cfg.layers, cfg.heads, cfg.ff = g.hidden, g.layers, g.heads, g.ff
    cfg.n_text_tokens, cfg.n_audio_tokens = g.n_text_tokens, g.n_audio_tokens
    cfg.start_audio_token, cfg.stop_audio_token = g.start_audio_token, g.stop_audio_token
    cfg.max_audio_tokens, cfg.max_text_tokens, cfg.n_cond_latents = g.max_audio_tokens, g.max_text_tokens, g.n_cond_latents
    cfg.ln_eps = g.ln_eps
    cfg.voc_in_dim, cfg.voc_init_ch, cfg.voc_n_up = v.in_dim, v.init_ch, len(v.up_rates)
    for i, (r, k) in enumerate(zip(v.up_rates, v.up_kernels)):
        cfg.voc_up_rates[i], cfg.voc_up_kernels[i] = r, k
    cfg.voc_n_rb = len(v.rb_kernels)
    for i, k in enumerate(v.rb_kernels):
        cfg.voc_rb_kernels[i] = k
    for i, d in enumerate(v.rb_dilations):
        cfg.voc_rb_dilations[i] = d
    cfg.d_vector = v.d_vector
    cfg.code_stride, cfg.output_hop_length = v.code_stride, v.output_hop_length
    cfg.input_sample_rate, cfg.output_sample_rate = v.input_sample_rate, v.output_sample_rate
    cfg.n_mels, cfg.cond_blocks, cfg.perceiver_depth = c.n_mels, c.cond_blocks, c.perceiver_depth
    cfg.perceiver_heads, cfg.perceiver_dim_head, cfg.perceiver_ff_mult = c.perceiver_heads, c.perceiver_dim_head, c.perceiver_ff_mult
    for i in range(4):
        cfg.spk_layers[i], cfg.spk_filters[i] = c.spk_layers[i], c.spk_filters[i]
    cfg.spk_mels, cfg.spk_proj = c.spk_mels, c.spk_proj
    return cfg


@dataclass
class Sampling:
    temperature: float = 0.75
    top_p: float = 0.85
    top_k: int = 50
    repetition_penalty: float = 5.0
    max_tokens: int = 605
    stop_token: int = 1025
    seed: int = 0
    seq_seed: int = 0
    vocode: bool = True
    priority: int = 0
    early_tokens: int = 0          # > 0: stream the chunk's audio as partial results, first piece after n tokens (include/xtts_b200.h)

    def c(self) -> XttsSampling:
        s = XttsSampling()
        s.temperature, s.top_p, s.repetition_penalty = self.temperature, self.top_p, self.repetition_penalty
        s.top_k, s.max_tokens, s.stop_token = self.top_k, self.max_tokens, self.stop_token
        s.seed, s.seq_seed, s.vocode = self.seed, self.seq_seed, 1 if self.vocode else 0
        s.priority = self.priority
        s.early_tokens = max(0, int(self.early_tokens))
        return s


class NativeEngine:
    """One engine = one GPU.  Thin, allocation-free wrapper over the C ABI."""

    def __init__(self, dims: XTTSDims, device: int = 0, precision: int = PRECISION_FP32, max_batch: int = 64,
                 max_speakers: int = 16):
        self.lib = load_library()
        self.dims = dims
        self.cfg = make_config(dims, device, precision, max_batch, max_speakers)
        self.precision = precision
        self.max_batch = max_batch
        h = C.c_void_p()
        rc = self.lib.xtts_create(C.byref(self.cfg), C.byref(h))
        if rc != 0:
            raise NativeError(f"xtts_create failed ({rc}): {self.lib.xtts_last_error().decode()}")
        self.h = h

    def _chk(self, rc: int, what: str):
        if rc != 0:
            raise NativeError(f"{what} failed ({rc}): {self.lib.xtts_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.xtts_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def load_state(self, *states: Dict[str, "object"]):
        for st in states:
            for name, t in st.items():
                a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
                a = _f32(a)
                shape = (C.c_int64 * max(1, a.ndim))(*a.shape) if a.ndim else (C.c_int64 * 1)(1)
                self._chk(self.lib.xtts_load_weight(self.h, name.encode(), _fp(a), shape, max(1, a.ndim) if a.ndim else 1),
                          f"load_weight({name})")
        self._chk(self.lib.xtts_finalize_weights(self.h), "finalize_weights")

    # ---- speakers
    def set_speaker(self, slot: int, cond_latents, d_vector):
        c, g = _f32(cond_latents).reshape(-1), _f32(d_vector).reshape(-1)
        assert c.size == self.dims.gpt.n_cond_latents * self.dims.gpt.hidden and g.size == self.dims.voc.d_vector
        self._chk(self.lib.xtts_set_speaker(self.h, slot, _fp(c), _fp(g)), "set_speaker")

    def get_speaker(self, slot: int) -> Tuple[np.ndarray, np.ndarray]:
        c = np.empty((self.dims.gpt.n_cond_latents, self.dims.gpt.hidden), np.float32)
        g = np.empty((self.dims.voc.d_vector,), np.float32)
        self._chk(self.lib.xtts_get_speaker(self.h, slot, _fp(c), _fp(g)), "get_speaker")
        return c, g

    def condition(self, slot: int, wav22k, wav16k, gpt_cond_len: int = 30, gpt_cond_chunk_len: int = 4):
        a, b = _f32(wav22k).reshape(-1), _f32(wav16k).reshape(-1)
        self._chk(self.lib.xtts_condition(self.h, slot, _fp(a), a.size, _fp(b), b.size, gpt_cond_len, gpt_cond_chunk_len),
                  "condition")

    # ---- generation
    def submit(self, seq_id: int, text_ids, speaker_slot: int, sp: Sampling):
        t = _i32(text_ids)
        cs = sp.c()
        self._chk(self.lib.xtts_submit(self.h, seq_id, _ip(t), t.size, speaker_slot, C.byref(cs)), "submit")

    def cancel(self, seq_id: int):
        self._chk(self.lib.xtts_cancel(self.h, seq_id), "cancel")

    def poll(self, timeout_ms: int = 1000) -> Optional[XttsResult]:
        r = XttsResult()
        rc = self.lib.xtts_poll(self.h, C.byref(r), timeout_ms)
        if rc < 0:
            self._chk(rc, "poll")
        return r if rc == 1 else None

    def fetch(self, r: XttsResult, want_wav: bool = True, want_latents: bool = False):
        toks = np.empty((max(1, r.n_tokens),), np.int32)
        wav = np.empty((r.n_samples,), np.float32) if (want_wav and r.n_samples > 0) else None
        lat = np.empty((r.n_tokens, self.dims.gpt.hidden), np.float32) if want_latents else None
        self._chk(self.lib.xtts_fetch(self.h, r.seq_id, _ip(toks), _fp(wav), _fp(lat)), "fetch")
        return toks[: r.n_tokens], wav, lat

    def set_option(self, key: str, value: int):
        self._chk(self.lib.xtts_set_option(self.h, key.encode(), value), f"set_option({key})")

    def stats(self) -> XttsStats:
        s = XttsStats()
        self._chk(self.lib.xtts_get_stats(self.h, C.byref(s)), "get_stats")
        return s

    def sync(self):
        self._chk(self.lib.xtts_sync(self.h), "sync")

    def timer_start(self):
        """CUDA event on the engine stream (call with the engine idle)."""
        self._chk(self.lib.xtts_device_timer(self.h, 0, None), "device_timer(start)")

    def timer_stop_ms(self) -> float:
        """Second event behind everything submitted so far; milliseconds on the device clock since timer_start()."""
        ms = C.c_double(0.0)
        self._chk(self.lib.xtts_device_timer(self.h, 1, C.byref(ms)), "device_timer(stop)")
        return float(ms.value)

    def trace_start(self):
        rc = self.lib.xtts_debug_trace(self.h, 1, None, 0)
        if rc < 0:
            self._chk(rc, "debug_trace(start)")

    def trace_stop(self, cap: int = 1 << 20) -> np.ndarray:
        """-> [n, 4] int64: (ns, kernel id, phase, last-CTA flag) sorted by time; grid size in column 4 of the raw word"""
        buf = np.zeros((cap, 2), np.uint64)
        n = self.lib.xtts_debug_trace(self.h, 0, buf.ctypes.data_as(C.POINTER(C.c_uint64)), cap)
        if n < 0:
            self._chk(n, "debug_trace(stop)")
        b = buf[:n]
        out = np.stack([b[:, 0].astype(np.int64), (b[:, 1] >> np.uint64(32) & np.uint64(0xFF)).astype(np.int64),
                        (b[:, 1] & np.uint64(0xFF)).astype(np.int64), (b[:, 1] >> np.uint64(8) & np.uint64(1)).astype(np.int64),
                        (b[:, 1] >> np.uint64(40)).astype(np.int64)], axis=1)
        return out[np.argsort(out[:, 0], kind="stable")]

    def kernel_profile(self) -> Dict[str, dict]:
        """{family: {ms, flops, bytes, launches}} accumulated since option "profile" was switched on."""
        p = XttsKernelProfile()
        self._chk(self.lib.xtts_get_kernel_profile(self.h, C.byref(p)), "get_kernel_profile")
        out = {}
        for i in range(p.n):
            if p.launches[i]:
                out[bytes(p.name[i]).split(b"\0")[0].decode()] = dict(ms=p.ms[i], flops=p.flops[i], bytes=p.bytes[i],
                                                                    launches=int(p.launches[i]))
        return out

    def run_batch(self, jobs, timeout_s: float = 600.0, want_wav: bool = True, want_latents: bool = False):
        """jobs: iterable of (seq_id, text_ids, speaker_slot, Sampling).  Returns {seq_id: (result, tokens, wav, lat)}.
        want_wav: True / False, or a set of seq ids whose waveforms are copied out (the others' wav is None)."""
        import time
        wav_ids = None if isinstance(want_wav, bool) else frozenset(want_wav)

        def wants_wav(sid):
            return want_wav if wav_ids is None else sid in wav_ids
        n = 0
        # batch submit: the scheduler admits nothing until the whole batch is queued, so admission waves (and with
        # them which chunks finish together and share a vocoder launch) do not depend on host timing
        self.set_option("hold_admission", 1)
        try:
            for sid, ids, spk, sp in jobs:
                self.submit(sid, ids, spk, sp)
                n += 1
        finally:
            self.set_option("hold_admission", 0)
        out, partials = {}, {}
        t_end = time.time() + timeout_s
        while len(out) < n:
            r = self.poll(1000)
            if r is None:
                if time.time() > t_end:
                    raise NativeError("run_batch timed out")
                continue
            if r.status < 0:
                self.lib.xtts_fetch(self.h, r.seq_id, None, None, None)      # releases the failed chunk's native buffers
                raise NativeError(f"sequence {r.seq_id} failed ({r.status}): {self.lib.xtts_last_error().decode()}")
            if r.status > 0:                 # partial piece (Sampling.early_tokens): kept, in order, next to the final result
                ptoks, pwav, _ = self.fetch(r, wants_wav(r.seq_id), False)
                partials.setdefault(r.seq_id, []).append((r, ptoks, pwav))
                continue
            toks, wav, lat = self.fetch(r, wants_wav(r.seq_id), want_latents)
            out[r.seq_id] = (r, toks, wav, lat)
        self.last_partials = partials        # {seq_id: [(result, tokens, wav), ...]} of the batch just run, oldest first
        return out


    # ---- synchronous single-stage entry points (parity tests)
    def vocode(self, latents, speaker_slot: int, stage: Optional[str] = None, stage_shape: Optional[Tuple[int, ...]] = None):
        lat = _f32(latents)
        T = lat.shape[0]
        ns = self.dims.voc.n_samples(T)
        wav = np.empty((ns,), np.float32)
        n_out = C.c_int32(0)
        st_arr = np.zeros(stage_shape, np.float32) if stage else None
        self._chk(self.lib.xtts_vocode(self.h, _fp(lat), T, speaker_slot, _fp(wav), C.byref(n_out),
                                       stage.encode() if stage else None, _fp(st_arr), st_arr.size if stage else 0), "vocode")
        assert n_out.value == ns, (n_out.value, ns)
        return (wav, st_arr) if stage else wav

    def vocode_window(self, latents, speaker_slot: int, z0: int, nz: int) -> np.ndarray:
        """z-frames [z0, z0 + nz) of the chunk as a window of its own -> nz * hop samples (include/xtts_b200.h)."""
        lat = _f32(latents)
        wav = np.empty((nz * self.dims.voc.hop,), np.float32)
        self._chk(self.lib.xtts_vocode_window(self.h, _fp(lat), lat.shape[0], speaker_slot, z0, nz, _fp(wav)), "vocode_window")
        return wav

    def gpt_prefill(self, text_ids, speaker_slot: int, audio_tokens=(), want_hidden: bool = False):
        g = self.dims.gpt
        t, a = _i32(text_ids), _i32(list(audio_tokens))
        n = max(1, a.size)
        rows = g.n_cond_latents + t.size + 1 + max(0, a.size - 1)
        hid = np.empty((rows, g.hidden), np.float32) if want_hidden else None
        logits = np.empty((n, g.n_audio_tokens), np.float32)
        lat = np.empty((n, g.hidden), np.float32)
        self._chk(self.lib.xtts_gpt_prefill(self.h, _ip(t), t.size, speaker_slot, _ip(a) if a.size else None, a.size,
                                            _fp(hid), _fp(logits), _fp(lat)), "gpt_prefill")
        return hid, logits, lat

    def gpt_teacher_forced(self, text_ids, speaker_slot: int, forced_tokens, sp: Sampling):
        g = self.dims.gpt
        t, f = _i32(text_ids), _i32(forced_tokens)
        n = f.size
        logits = np.empty((n, g.n_audio_tokens), np.float32)
        lat = np.empty((n, g.hidden), np.float32)
        sampled = np.empty((n,), np.int32)
        cs = sp.c()
        self._chk(self.lib.xtts_gpt_teacher_forced(self.h, _ip(t), t.size, speaker_slot, _ip(f), n, C.byref(cs),
                                                   _fp(logits), _fp(lat), _ip(sampled)), "gpt_teacher_forced")
        return logits, lat, sampled

    def debug_gemm(self, mode: int, A, W, bias=None, resid=None, gelu: bool = False, iters: int = 0):
        A, W = _f32(A), _f32(W)
        M, K = A.shape
        N = W.shape[0]
        b = _f32(bias) if bias is not None else None
        r = _f32(resid) if resid is not None else None
        out = np.empty((M, N), np.float32)
        ms = C.c_float(0)
        self._chk(self.lib.xtts_debug_gemm(self.h, mode, _fp(A), _fp(W), _fp(b), _fp(r), _fp(out), M, N, K,
                                           1 if gelu else 0, iters, C.byref(ms)), "debug_gemm")
        return out, ms.value

    def debug_sample(self, logits, seen, sp: Sampling, step: int = 0):
        lg = _f32(logits)
        Bn, V = lg.shape
        sn = np.ascontiguousarray(np.asarray(seen, dtype=np.uint8)) if seen is not None else None
        out = np.empty((Bn,), np.int32)
        cs = sp.c()
        self._chk(self.lib.xtts_debug_sample(self.h, _fp(lg), sn.ctypes.data_as(C.POINTER(C.c_uint8)) if sn is not None else None,
                                             Bn, V, C.byref(cs), step, _ip(out)), "debug_sample")
        return out
