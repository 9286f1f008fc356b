"""CPU parity oracle (TEST INFRASTRUCTURE ONLY).

ctypes front-end to ``oracle/liboracle.so`` (built from ``oracle.c`` by ``oracle/Makefile``),
the C restatement of the reference's futuredsp / block arithmetic.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this package; nothing under ``futuresdr_b200/`` does.

Status codes follow ``futuredsp::ComputationStatus`` (crates/futuredsp/src/lib.rs:33-45):
0 InsufficientInput, 1 InsufficientOutput, 2 BothSufficient.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")

INSUFFICIENT_INPUT, INSUFFICIENT_OUTPUT, BOTH_SUFFICIENT = 0, 1, 2


def build(force: bool = False) -> str:
    """Compile liboracle.so if missing (gcc only; seconds).  An existing library is loaded as it is:
    the tests and bench.py may run from a read-only tree, and ``__graft_entry__.build()`` remakes the
    library whenever its sources change."""
    if force or not os.path.exists(_SO):
        subprocess.run(["make", "-C", _HERE, "-s", "clean", "all"], check=True)
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _declare(_lib)
    return _lib


_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_szp = C.POINTER(C.c_size_t)


def _declare(L):
    for name in ("orc_fir_f32_f32", "orc_fir_c32_f32", "orc_fir_c32_c32"):
        f = getattr(L, name)
        f.restype = C.c_int
        f.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t, _f32p, C.c_size_t, _szp, _szp]
    L.orc_fir_f64_f64.restype = C.c_int
    L.orc_fir_f64_f64.argtypes = [_f64p, C.c_size_t, _f64p, C.c_size_t, _f64p, C.c_size_t, _szp, _szp]
    for name in ("orc_decim_f32_f32", "orc_decim_c32_f32", "orc_decim_c32_c32"):
        f = getattr(L, name)
        f.restype = C.c_int
        f.argtypes = [_f32p, C.c_size_t, C.c_size_t, _f32p, C.c_size_t, _f32p, C.c_size_t, _szp, _szp]
    for name in ("orc_resamp_f32_f32", "orc_resamp_c32_f32"):
        f = getattr(L, name)
        f.restype = C.c_int
        f.argtypes = [_f32p, C.c_size_t, C.c_size_t, C.c_size_t, _f32p, C.c_size_t, _f32p,
                      C.c_size_t, _szp, _szp]
    L.orc_fir_c32_f32_exact.restype = None
    L.orc_fir_c32_f32_exact.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t, C.c_size_t, _f64p]
    L.orc_besseli0.restype = C.c_double
    L.orc_besseli0.argtypes = [C.c_double]
    L.orc_window_kaiser.restype = None
    L.orc_window_kaiser.argtypes = [C.c_size_t, C.c_double, _f64p]
    L.orc_firdes_lowpass.restype = None
    L.orc_firdes_lowpass.argtypes = [C.c_double, _f64p, C.c_size_t, _f64p]
    L.orc_kaiser_beta.restype = C.c_double
    L.orc_kaiser_beta.argtypes = [C.c_double]
    L.orc_kaiser_num_taps.restype = C.c_size_t
    L.orc_kaiser_num_taps.argtypes = [C.c_double, C.c_double]
    L.orc_kaiser_lowpass.restype = C.c_size_t
    L.orc_kaiser_lowpass.argtypes = [C.c_double, C.c_double, C.c_double, _f64p, C.c_size_t]
    L.orc_kaiser_multirate.restype = C.c_size_t
    L.orc_kaiser_multirate.argtypes = [C.c_size_t, C.c_size_t, C.c_size_t, C.c_double, _f64p, C.c_size_t]
    L.orc_fft_block_c32.restype = C.c_size_t
    L.orc_fft_block_c32.argtypes = [C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float, _f32p,
                                    C.c_size_t, _f32p, C.c_size_t]
    L.orc_apply_quad_demod.restype = None
    L.orc_apply_quad_demod.argtypes = [_f32p, C.c_size_t, _f32p, _f32p]
    L.orc_apply_scale_f32.restype = None
    L.orc_apply_scale_f32.argtypes = [_f32p, C.c_size_t, C.c_float, _f32p]
    L.orc_apply_norm_sqr.restype = None
    L.orc_apply_norm_sqr.argtypes = [_f32p, C.c_size_t, _f32p]
    L.orc_pfbarb_new.restype = C.c_void_p
    L.orc_pfbarb_new.argtypes = [C.c_float, _f32p, C.c_size_t, C.c_size_t]
    L.orc_pfbarb_free.restype = None
    L.orc_pfbarb_free.argtypes = [C.c_void_p]
    L.orc_pfbarb_work.restype = None
    L.orc_pfbarb_work.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_size_t, _szp, _szp,
                                  C.POINTER(C.c_int)]
    L.orc_rotator_incr.restype = None
    L.orc_rotator_incr.argtypes = [C.c_float, _f32p]
    L.orc_rotator_rotate.restype = None
    L.orc_rotator_rotate.argtypes = [_f32p, C.c_size_t, _f32p, _f32p, _f32p]
    L.orc_xlating_taps.restype = None
    L.orc_xlating_taps.argtypes = [_f32p, C.c_size_t, C.c_float, C.c_float, _f32p]
    L.orc_max_threads.restype = C.c_int
    for name in ("orc_fir_c32_f32_mt", "orc_fir_c32_f32_fast_mt"):
        f = getattr(L, name)
        f.restype = None
        f.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t, _f32p, C.c_int]


def _p32(a):
    return a.ctypes.data_as(_f32p)


def _p64(a):
    return a.ctypes.data_as(_f64p)


def _as(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _nitems(a: np.ndarray) -> int:
    return a.size


def _filter(fn_real, fn_c32f, fn_c32c, taps, x, out_cap, extra=()):
    """Dispatch on dtypes like the Rust trait impls do. Returns (consumed, produced, status, out)."""
    x = np.ascontiguousarray(x)
    taps = np.ascontiguousarray(taps)
    cplx_in = np.iscomplexobj(x)
    cplx_tap = np.iscomplexobj(taps)
    n_in = x.size
    ntaps = taps.size
    if out_cap is None:
        out_cap = n_in
    c, p = C.c_size_t(0), C.c_size_t(0)
    if not cplx_in:
        assert not cplx_tap and fn_real is not None
        xi, tp = _as(x, np.float32), _as(taps, np.float32)
        out = np.zeros(max(out_cap, 1), np.float32)
        st = fn_real(_p32(tp), ntaps, *extra, _p32(xi), n_in, _p32(out), out_cap, C.byref(c), C.byref(p))
        return c.value, p.value, st, out[: p.value].copy()
    xi = _as(x, np.complex64)
    out = np.zeros(max(out_cap, 1), np.complex64)
    if cplx_tap:
        assert fn_c32c is not None
        tp = _as(taps, np.complex64)
        st = fn_c32c(_p32(tp.view(np.float32)), ntaps, *extra, _p32(xi.view(np.float32)), n_in,
                     _p32(out.view(np.float32)), out_cap, C.byref(c), C.byref(p))
    else:
        tp = _as(taps, np.float32)
        st = fn_c32f(_p32(tp), ntaps, *extra, _p32(xi.view(np.float32)), n_in,
                     _p32(out.view(np.float32)), out_cap, C.byref(c), C.byref(p))
    return c.value, p.value, st, out[: p.value].copy()


def fir(taps, x, out_cap=None):
    """FirFilter::filter (crates/futuredsp/src/fir.rs:52-91)."""
    L = lib()
    return _filter(L.orc_fir_f32_f32, L.orc_fir_c32_f32, L.orc_fir_c32_c32, taps, x, out_cap)


def fir_f64(taps, x, out_cap=None):
    L = lib()
    x = _as(x, np.float64); taps = _as(taps, np.float64)
    if out_cap is None:
        out_cap = x.size
    out = np.zeros(max(out_cap, 1), np.float64)
    c, p = C.c_size_t(0), C.c_size_t(0)
    st = L.orc_fir_f64_f64(_p64(taps), taps.size, _p64(x), x.size, _p64(out), out_cap, C.byref(c), C.byref(p))
    return c.value, p.value, st, out[: p.value].copy()


def decim_fir(taps, decim, x, out_cap=None):
    """DecimatingFirFilter::filter (decimating_fir.rs:53-95)."""
    L = lib()
    return _filter(L.orc_decim_f32_f32, L.orc_decim_c32_f32, L.orc_decim_c32_c32, taps, x, out_cap,
                   extra=(int(decim),))


def resamp_fir(taps, interp, decim, x, out_cap=None):
    """PolyphaseResamplingFir::filter (polyphase_resampling_fir.rs:70-124)."""
    L = lib()
    assert len(taps) % interp == 0, "ntaps % interp == 0 (polyphase_resampling_fir.rs:56)"
    if out_cap is None:
        out_cap = (np.asarray(x).size * interp) // decim + interp
    return _filter(L.orc_resamp_f32_f32, L.orc_resamp_c32_f32, None, taps, x, out_cap,
                   extra=(int(interp), int(decim)))


def fir_c32_exact(taps, x, n_out, decim=1):
    """f64-accumulated value of the same sums (arbiter, not a reference function)."""
    L = lib()
    xi = _as(x, np.complex64); tp = _as(taps, np.float32)
    out = np.zeros(n_out, np.complex128)
    L.orc_fir_c32_f32_exact(_p32(tp), tp.size, _p32(xi.view(np.float32)), n_out, decim,
                            _p64(out.view(np.float64)))
    return out


def besseli0(x):
    return lib().orc_besseli0(float(x))


def window_kaiser(n, beta):
    w = np.zeros(n, np.float64)
    lib().orc_window_kaiser(n, float(beta), _p64(w))
    return w


def firdes_lowpass(cutoff, window):
    window = _as(window, np.float64)
    t = np.zeros(window.size, np.float64)
    lib().orc_firdes_lowpass(float(cutoff), _p64(window), window.size, _p64(t))
    return t


def kaiser_lowpass(cutoff, transition_bw, max_ripple, dtype=np.float32):
    """firdes::kaiser::lowpass::<T> (firdes/basic.rs:310-321); T::from_f64 = dtype cast."""
    L = lib()
    n = L.orc_kaiser_lowpass(cutoff, transition_bw, max_ripple, None, 0)
    t = np.zeros(n, np.float64)
    L.orc_kaiser_lowpass(cutoff, transition_bw, max_ripple, _p64(t), n)
    return t.astype(dtype)


def kaiser_multirate(interp, decim, half_len, max_ripple, dtype=np.float32):
    """firdes::kaiser::multirate::<T> (firdes/basic.rs:412-442)."""
    L = lib()
    n = L.orc_kaiser_multirate(interp, decim, half_len, max_ripple, None, 0)
    t = np.zeros(n, np.float64)
    L.orc_kaiser_multirate(interp, decim, half_len, max_ripple, _p64(t), n)
    return t.astype(dtype)


def fft_block(x, n, inverse=False, fft_shift=False, normalize=None, out_cap=None):
    """Fft::work over everything available (src/blocks/fft.rs:160-221). Returns (m, out)."""
    xi = _as(x, np.complex64)
    if out_cap is None:
        out_cap = xi.size
    out = np.zeros(max(out_cap, 1), np.complex64)
    m = lib().orc_fft_block_c32(n, int(inverse), int(fft_shift), int(normalize is not None),
                                float(normalize or 0.0), _p32(xi.view(np.float32)), xi.size,
                                _p32(out.view(np.float32)), out_cap)
    return m, out[:m].copy()


def quad_demod(x, carry=(0.0, 0.0)):
    """Apply closure of examples/fm-receiver/src/main.rs:99-104. Returns (out, carry)."""
    xi = _as(x, np.complex64)
    out = np.zeros(xi.size, np.float32)
    cr = np.array(carry, np.float32)
    lib().orc_apply_quad_demod(_p32(xi.view(np.float32)), xi.size, _p32(out), _p32(cr))
    return out, (float(cr[0]), float(cr[1]))


def scale_f32(x, k):
    xi = _as(x, np.float32)
    out = np.zeros(xi.size, np.float32)
    lib().orc_apply_scale_f32(_p32(xi), xi.size, float(k), _p32(out))
    return out


def norm_sqr(x):
    xi = _as(x, np.complex64)
    out = np.zeros(xi.size, np.float32)
    lib().orc_apply_norm_sqr(_p32(xi.view(np.float32)), xi.size, _p32(out))
    return out


class PfbArb:
    """PfbArbResampler state machine (src/blocks/pfb/arb_resampler.rs:90-231)."""

    def __init__(self, rate, taps, num_filters):
        taps = _as(taps, np.float32)
        assert rate > 0 and taps.size >= num_filters and num_filters != 0
        self.rate = np.float32(rate)
        self._h = lib().orc_pfbarb_new(float(rate), _p32(taps), taps.size, num_filters)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_pfbarb_free(self._h)
            self._h = None

    def work(self, x, out_cap):
        """One Kernel::work call: returns (consumed, produced, call_again, out)."""
        xi = _as(x, np.complex64)
        out = np.zeros(max(out_cap, 1) + 8, np.complex64)
        c, p, ca = C.c_size_t(0), C.c_size_t(0), C.c_int(0)
        lib().orc_pfbarb_work(self._h, _p32(xi.view(np.float32)), xi.size,
                              _p32(out.view(np.float32)), out_cap, C.byref(c), C.byref(p), C.byref(ca))
        return c.value, p.value, bool(ca.value), out[: p.value].copy()

    def run(self, x, out_cap_per_call=1 << 20):
        """Mocker-style loop (src/runtime/mocker.rs:159-190): call work until input is drained."""
        xi = _as(x, np.complex64)
        outs, pos = [], 0
        while True:
            c, p, ca, o = self.work(xi[pos:], out_cap_per_call)
            pos += c
            outs.append(o)
            if c == 0 and p == 0 and not ca:
                break
        return np.concatenate(outs) if outs else np.zeros(0, np.complex64)


class Rotator:
    """futuredsp::Rotator (crates/futuredsp/src/rotator.rs:13-48)."""

    def __init__(self, phase_incr):
        self.incr = np.zeros(2, np.float32)
        lib().orc_rotator_incr(float(np.float32(phase_incr)), _p32(self.incr))
        self.phase = np.array([1.0, 0.0], np.float32)

    def rotate(self, x):
        xi = _as(x, np.complex64)
        out = np.zeros(xi.size, np.complex64)
        lib().orc_rotator_rotate(_p32(xi.view(np.float32)), xi.size, _p32(out.view(np.float32)),
                                 _p32(self.incr), _p32(self.phase))
        return out


class PfbChannelizer:
    """PfbChannelizer state machine (src/blocks/pfb/channelizer.rs:88-223)."""

    def __init__(self, num_channels, taps, oversample_rate=1.0):
        taps = _as(taps, np.float32)
        assert num_channels > 2 and taps.size >= num_channels
        assert oversample_rate != 0 and (num_channels % oversample_rate) == 0
        L = lib()
        L.orc_chan_new.restype = C.c_void_p
        L.orc_chan_new.argtypes = [C.c_size_t, _f32p, C.c_size_t, C.c_float]
        L.orc_chan_free.restype = None
        L.orc_chan_free.argtypes = [C.c_void_p]
        L.orc_chan_work.restype = None
        L.orc_chan_work.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_size_t, C.c_size_t, _szp, _szp,
                                    C.POINTER(C.c_int)]
        self.N = num_channels
        self.D = int(np.float32(num_channels) / np.float32(oversample_rate))
        self._h = L.orc_chan_new(num_channels, _p32(taps), taps.size, float(oversample_rate))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_chan_free(self._h)
            self._h = None

    def work(self, x, out_cap):
        """One Kernel::work call -> (consumed, produced_per_channel, call_again, out[N, produced])."""
        xi = _as(x, np.complex64)
        out = np.zeros((self.N, max(out_cap, 1)), np.complex64)
        c, p, ca = C.c_size_t(0), C.c_size_t(0), C.c_int(0)
        lib().orc_chan_work(self._h, _p32(xi.view(np.float32)), xi.size, _p32(out.view(np.float32).reshape(-1)),
                            max(out_cap, 1), out_cap, C.byref(c), C.byref(p), C.byref(ca))
        return c.value, p.value, bool(ca.value), out[:, : p.value].copy()

    def run(self, x, out_cap_per_call=1 << 16):
        """Mocker-style loop: call work() until nothing more can be consumed."""
        xi = _as(x, np.complex64)
        outs, pos = [], 0
        for _ in range(1 << 20):
            c, p, ca, o = self.work(xi[pos:], out_cap_per_call)
            pos += c
            outs.append(o)
            if c == 0 and p == 0 and not ca:
                break
        return np.concatenate(outs, axis=1)


class PfbSynthesizer:
    """PfbSynthesizer state machine (src/blocks/pfb/synthesizer.rs:52-144)."""

    def __init__(self, num_channels, taps):
        taps = _as(taps, np.float32)
        L = lib()
        L.orc_synth_new.restype = C.c_void_p
        L.orc_synth_new.argtypes = [C.c_size_t, _f32p, C.c_size_t]
        L.orc_synth_free.restype = None
        L.orc_synth_free.argtypes = [C.c_void_p]
        L.orc_synth_work.restype = None
        L.orc_synth_work.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, _f32p, C.c_size_t, _szp, _szp]
        self.N = num_channels
        self._h = L.orc_synth_new(num_channels, _p32(taps), taps.size)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_synth_free(self._h)
            self._h = None

    def work(self, x, out_cap):
        """x: [N, n] channel-major inputs. Returns (consumed_per_channel, produced, out)."""
        xi = np.ascontiguousarray(x, dtype=np.complex64)
        assert xi.shape[0] == self.N
        out = np.zeros(max(out_cap, self.N) + self.N, np.complex64)
        c, p = C.c_size_t(0), C.c_size_t(0)
        lib().orc_synth_work(self._h, _p32(xi.view(np.float32).reshape(-1)), xi.shape[1], xi.shape[1],
                             _p32(out.view(np.float32)), out_cap, C.byref(c), C.byref(p))
        return c.value, p.value, out[: p.value].copy()


class MovingAvg:
    """MovingAvg<WIDTH> (src/blocks/moving_avg.rs:24-116)."""

    def __init__(self, width, decay_factor, history_size):
        assert 0.0 <= decay_factor <= 1.0, "decay_factor must be in [0, 1]"
        self.width, self.decay, self.history = int(width), float(np.float32(decay_factor)), int(history_size)
        self.avg = np.zeros(self.width, np.float32)
        self.i = C.c_size_t(0)
        L = lib()
        L.orc_mavg_work.restype = None
        L.orc_mavg_work.argtypes = [_f32p, _szp, C.c_size_t, C.c_float, C.c_size_t, _f32p, C.c_size_t, _f32p,
                                    C.c_size_t, _szp, _szp]

    def work(self, x, out_cap):
        xi = _as(x, np.float32)
        out = np.zeros(max(out_cap, 1), np.float32)
        c, p = C.c_size_t(0), C.c_size_t(0)
        lib().orc_mavg_work(_p32(self.avg), C.byref(self.i), self.width, self.decay, self.history, _p32(xi),
                            xi.size, _p32(out), out_cap, C.byref(c), C.byref(p))
        return c.value, p.value, out[: p.value].copy()


def xlating_taps(taps, offset, sample_rate):
    """Band-pass taps of XlatingFir (src/blocks/xlating_fir.rs:80-86)."""
    t = _as(taps, np.float32)
    out = np.zeros(t.size, np.complex64)
    lib().orc_xlating_taps(_p32(t), t.size, float(np.float32(offset)), float(np.float32(sample_rate)),
                           _p32(out.view(np.float32)))
    return out


def xlating_fir(taps, decimation, offset, sample_rate, x, chunks=None):
    """XlatingFir::work over a stream (src/blocks/xlating_fir.rs:105-126): decimating FIR with the
    band-pass taps, then the rotator at the output rate.  Returns the whole output."""
    bpf = xlating_taps(taps, offset, sample_rate)
    rot = Rotator(np.float32(-6.28318530717958647692) * np.float32(offset) * np.float32(decimation)
                  / np.float32(sample_rate))
    _, _, _, y = decim_fir(bpf, decimation, x, np.asarray(x).size)
    return rot.rotate(y)


def max_threads():
    return lib().orc_max_threads()


def fir_c32_f32_mt(taps, x, threads, fast=False, out=None):
    """All-core strict-order (or nightly/fast-math) c32 x f32 FIR for the CPU baseline."""
    L = lib()
    xi = _as(x, np.complex64); tp = _as(taps, np.float32)
    n = max(xi.size + 1 - tp.size, 0)
    if out is None:
        out = np.empty(n, np.complex64)
    fn = L.orc_fir_c32_f32_fast_mt if fast else L.orc_fir_c32_f32_mt
    fn(_p32(tp), tp.size, _p32(xi.view(np.float32)), xi.size, _p32(out.view(np.float32)), int(threads))
    return out
