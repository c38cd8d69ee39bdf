"""ctypes front-ends for the two CPU checkers.  TEST INFRASTRUCTURE -- never imported by csdr_b200.

* ``Oracle``  -> oracle/liboracle.so        our strict-IEEE C restatement (oracle.c)
* ``Ref``     -> oracle/_ref/libcsdr_ref.so the unmodified reference compiled from /root/reference
                                             (``make -C oracle ref``; travels to the GPU box as a binary)

Both expose the same numpy-level API so a test can be parametrised over them.
complex samples are numpy complex64 arrays (= interleaved float32 I,Q = reference ``complexf``).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "liboracle.so"
REF_SO = HERE / "_ref" / "libcsdr_ref.so"
REF_CLI = HERE / "_ref" / "csdr_ref"

WINDOWS = {"BOXCAR": 0, "BLACKMAN": 1, "HAMMING": 2}


def build(ref: bool | None = None) -> None:
    """Compile the checkers.  ``ref`` defaults to "only where $CSDR_REFERENCE names a readable csdr source tree"; without it
    the tests compare against the reference outputs stored under tests/golden/."""
    subprocess.run(["make", "-s", "-C", str(HERE), "oracle"], check=True)
    src = os.environ.get("CSDR_REFERENCE", "")
    if ref is None:
        ref = bool(src) and os.access(src, os.R_OK | os.X_OK) and os.path.isfile(os.path.join(src, "libcsdr.c"))
    if ref:
        subprocess.run(["make", "-s", "-C", str(HERE), "ref"] + ([f"REF={src}"] if src else []), check=True)


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class _CF(C.Structure):
    _fields_ = [("i", C.c_float), ("q", C.c_float)]


class _Shift(C.Structure):
    _fields_ = [("sindelta", C.c_float), ("cosdelta", C.c_float), ("rate", C.c_float)]


class _DShiftStatus(C.Structure):
    _fields_ = [("decimation_remain", C.c_int), ("starting_phase", C.c_float), ("output_size", C.c_int)]


def _c64(a):
    a = np.ascontiguousarray(a, dtype=np.complex64)
    return a


# ======================================================================================================
class Oracle:
    """Binding of oracle/liboracle.so (see oracle.h)."""

    name = "oracle"

    class _FracDec(C.Structure):
        _fields_ = [("where", C.c_float), ("input_processed", C.c_int), ("output_size", C.c_int),
                    ("num_poly_points", C.c_int), ("xifirst", C.c_int), ("xilast", C.c_int),
                    ("rate", C.c_float), ("denom", C.c_float * 64),
                    ("taps", C.POINTER(C.c_float)), ("taps_length", C.c_int)]

    class _Agc(C.Structure):
        _fields_ = [("peak_1", C.c_float), ("peak_2", C.c_float), ("reference", C.c_float),
                    ("last_gain", C.c_float), ("block", C.c_int)]

    class _Ddc(C.Structure):
        _fields_ = [(n, C.c_int) for n in ("pre_decimation", "post_decimation", "taps_length", "taps_min_length",
                                           "overlap_length", "fft_size", "fft_inv_size", "input_size",
                                           "post_input_size")] + \
                   [("pre_shift", C.c_float), ("startbin", C.c_int), ("v", C.c_int), ("offsetbin", C.c_int),
                    ("post_shift", C.c_float), ("scrap", C.c_int), ("dsadata", _Shift)]

    def __init__(self, path: Path = ORACLE_SO):
        if not path.exists():
            build(ref=False)
        L = self.L = C.CDLL(str(path))
        L.oracle_firdes_filter_len.argtypes = [C.c_float]
        L.oracle_window.argtypes = [C.c_int, C.c_float]; L.oracle_window.restype = C.c_float
        L.oracle_firdes_lowpass_f.argtypes = [C.POINTER(C.c_float), C.c_int, C.c_float, C.c_int]
        L.oracle_firdes_bandpass_c.argtypes = [C.POINTER(_CF), C.c_int, C.c_float, C.c_float, C.c_int]
        L.oracle_shift_addition_init.argtypes = [C.c_float]; L.oracle_shift_addition_init.restype = _Shift
        L.oracle_shift_addition_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, _Shift, C.c_float]
        L.oracle_shift_addition_cc.restype = C.c_float
        L.oracle_decimating_shift_addition_init.argtypes = [C.c_float, C.c_int]
        L.oracle_decimating_shift_addition_init.restype = _Shift
        L.oracle_decimating_shift_addition_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, _Shift, C.c_int, _DShiftStatus]
        L.oracle_decimating_shift_addition_cc.restype = _DShiftStatus
        L.oracle_fir_decimate_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_int, C.POINTER(C.c_float), C.c_int]
        L.oracle_fmdemod_quadri_cf.argtypes = [C.POINTER(_CF), C.POINTER(C.c_float), C.c_int, _CF]
        L.oracle_fmdemod_quadri_cf.restype = _CF
        L.oracle_fractional_decimator_ff_init.argtypes = [C.POINTER(self._FracDec), C.c_float, C.c_int, C.POINTER(C.c_float), C.c_int]
        L.oracle_fractional_decimator_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.POINTER(self._FracDec)]
        L.oracle_fastagc_ff.argtypes = [C.POINTER(self._Agc)] + [C.POINTER(C.c_float)] * 4
        L.oracle_deemphasis_wfm_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_float, C.c_int, C.c_float]
        L.oracle_deemphasis_wfm_ff.restype = C.c_float
        L.oracle_limit_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_float]
        L.oracle_deemphasis_nfm_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_float), C.c_int]
        fp = C.POINTER(C.c_float)
        L.oracle_precalculate_window.argtypes = [fp, C.c_int, C.c_int]
        L.oracle_apply_precalculated_window_c.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, fp]
        L.oracle_logpower_cf.argtypes = [C.POINTER(_CF), fp, C.c_int, C.c_float]
        L.oracle_accumulate_power_cf.argtypes = [C.POINTER(_CF), fp, C.c_int]
        L.oracle_log_ff.argtypes = [fp, fp, C.c_int, C.c_float]
        L.oracle_shift_unroll_init.argtypes = [C.c_float, C.c_int, fp, fp]; L.oracle_shift_unroll_init.restype = C.c_float
        L.oracle_shift_unroll_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, fp, fp, C.c_float, C.c_float]
        L.oracle_shift_unroll_cc.restype = C.c_float
        L.oracle_encode_ima_adpcm_i16_u8.argtypes = [C.POINTER(C.c_short), C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.oracle_compress_fft_adpcm_f_u8.argtypes = [fp, C.POINTER(C.c_ubyte), C.c_int]
        L.oracle_shift_table_init.argtypes = [fp, C.c_int]
        L.oracle_shift_table_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_float, fp, C.c_int, C.c_float, C.POINTER(C.c_int)]
        L.oracle_shift_table_cc.restype = C.c_float
        L.oracle_shift_math_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_float, C.c_float]; L.oracle_shift_math_cc.restype = C.c_float
        L.oracle_shift_addfast_init.argtypes = [C.c_float, fp]
        L.oracle_shift_addfast_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, fp, C.c_float]; L.oracle_shift_addfast_cc.restype = C.c_float
        L.oracle_dft_c2c.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_int]
        L.oracle_apply_fir_fft_cc.argtypes = [C.POINTER(_CF)] * 3 + [C.c_int, C.POINTER(_CF), C.c_int]
        L.oracle_fastddc_init.argtypes = [C.POINTER(self._Ddc), C.c_float, C.c_int, C.c_float]
        L.oracle_fastddc_make_taps_fft.argtypes = [C.POINTER(self._Ddc), C.c_float, C.c_int, C.c_int, C.POINTER(_CF)]
        L.oracle_fastddc_inv_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.POINTER(self._Ddc), C.POINTER(_CF), _DShiftStatus]
        L.oracle_fastddc_inv_cc.restype = _DShiftStatus

    # ---- conversions
    def convert_u8_f(self, x):
        x = np.ascontiguousarray(x, np.uint8); y = np.empty(x.size, np.float32)
        self.L.oracle_convert_u8_f(_p(x, C.c_ubyte), _p(y, C.c_float), x.size); return y

    def convert_s16_f(self, x):
        x = np.ascontiguousarray(x, np.int16); y = np.empty(x.size, np.float32)
        self.L.oracle_convert_s16_f(_p(x, C.c_short), _p(y, C.c_float), x.size); return y

    def convert_f_s16(self, x):
        x = np.ascontiguousarray(x, np.float32); y = np.empty(x.size, np.int16)
        self.L.oracle_convert_f_s16(_p(x, C.c_float), _p(y, C.c_short), x.size); return y

    # ---- filter design
    def firdes_filter_len(self, bw): return int(self.L.oracle_firdes_filter_len(bw))

    def firdes_lowpass_f(self, length, cutoff, window="HAMMING"):
        t = np.empty(length, np.float32)
        self.L.oracle_firdes_lowpass_f(_p(t, C.c_float), length, cutoff, WINDOWS[window]); return t

    def firdes_bandpass_c(self, length, lo, hi, window="HAMMING"):
        t = np.empty(length, np.complex64)
        self.L.oracle_firdes_bandpass_c(_p(t, _CF), length, lo, hi, WINDOWS[window]); return t

    # ---- shift
    def shift_addition_init(self, rate):
        d = self.L.oracle_shift_addition_init(rate); return (d.sindelta, d.cosdelta, d.rate)

    def shift_addition_cc(self, x, rate, phase=0.0, chunk=None):
        """Returns (y, final_phase).  ``chunk`` reproduces the CLI's <=1024-sample sub-calls (csdr.c:911-918)."""
        x = _c64(x); y = np.empty_like(x); d = self.L.oracle_shift_addition_init(rate)
        chunk = chunk or max(x.size, 1)
        for s in range(0, x.size, chunk):
            n = min(chunk, x.size - s)
            phase = self.L.oracle_shift_addition_cc(_p(x[s:], _CF), _p(y[s:], _CF), n, d, phase)
        return y, float(np.float32(phase))

    def decimating_shift_addition_cc(self, x, rate, decimation, remain=0, phase=0.0):
        x = _c64(x); y = np.empty(x.size // decimation + 2, np.complex64)
        d = self.L.oracle_decimating_shift_addition_init(rate, decimation)
        st = self.L.oracle_decimating_shift_addition_cc(_p(x, _CF), _p(y, _CF), x.size, d, decimation,
                                                        _DShiftStatus(remain, phase, 0))
        return y[:st.output_size].copy(), (st.decimation_remain, st.starting_phase)

    # ---- FIR
    def fir_decimate_cc(self, x, decimation, taps):
        x = _c64(x); taps = np.ascontiguousarray(taps, np.float32)
        y = np.empty(max(x.size // decimation + 1, 1), np.complex64)
        n = self.L.oracle_fir_decimate_cc(_p(x, _CF), _p(y, _CF), x.size, decimation, _p(taps, C.c_float), taps.size)
        return y[:n].copy()

    # ---- fmdemod
    def fmdemod_quadri_cf(self, x, last=0j):
        x = _c64(x); y = np.empty(x.size, np.float32)
        r = self.L.oracle_fmdemod_quadri_cf(_p(x, _CF), _p(y, C.c_float), x.size, _CF(np.float32(last.real), np.float32(last.imag)))
        return y, complex(r.i, r.q)

    # ---- fractional decimator (streamed block by block like csdr.c:1510-1522 when block is given)
    def fractional_decimator_ff(self, x, rate, num_poly_points=12, taps=None, block=None):
        x = np.ascontiguousarray(x, np.float32)
        tp = np.ascontiguousarray(taps, np.float32) if taps is not None else None
        d = self._FracDec()
        self.L.oracle_fractional_decimator_ff_init(C.byref(d), rate, num_poly_points,
                                                   _p(tp, C.c_float) if tp is not None else None,
                                                   tp.size if tp is not None else 0)
        return _stream_fracdec(lambda buf, out, n: self.L.oracle_fractional_decimator_ff(_p(buf, C.c_float), _p(out, C.c_float), n, C.byref(d)),
                               d, x, block)

    # ---- fastagc (streamed)
    def fastagc_ff(self, x, block=1024, reference=1.0):
        x = np.ascontiguousarray(x, np.float32); nblk = x.size // block
        st = self._Agc(0, 0, reference, 0, block)
        h1 = np.zeros(block, np.float32); h2 = np.zeros(block, np.float32); y = np.empty(nblk * block, np.float32)
        for b in range(nblk):
            self.L.oracle_fastagc_ff(C.byref(st), _p(h1, C.c_float), _p(h2, C.c_float),
                                     _p(x[b * block:], C.c_float), _p(y[b * block:], C.c_float))
        return y

    # ---- audio tail
    def deemphasis_wfm_ff(self, x, tau, sample_rate, last=0.0, block=None):
        x = np.ascontiguousarray(x, np.float32); y = np.empty_like(x); block = block or max(x.size, 1)
        for s0 in range(0, x.size, block):
            n = min(block, x.size - s0)
            last = self.L.oracle_deemphasis_wfm_ff(_p(x[s0:], C.c_float), _p(y[s0:], C.c_float), n, tau, sample_rate, last)
        return y, float(np.float32(last))

    def limit_ff(self, x, max_amplitude=1.0):
        x = np.ascontiguousarray(x, np.float32); y = np.empty_like(x)
        self.L.oracle_limit_ff(_p(x, C.c_float), _p(y, C.c_float), x.size, max_amplitude); return y

    def deemphasis_nfm_ff(self, x, taps):
        x = np.ascontiguousarray(x, np.float32); taps = np.ascontiguousarray(taps, np.float32); y = np.empty_like(x)
        n = self.L.oracle_deemphasis_nfm_ff(_p(x, C.c_float), _p(y, C.c_float), x.size, _p(taps, C.c_float), taps.size)
        return y[:n].copy()

    # ---- spectrum side path, shift_unroll
    def precalculate_window(self, size, window="HAMMING"):
        w = np.empty(size, np.float32); self.L.oracle_precalculate_window(_p(w, C.c_float), size, WINDOWS[window]); return w

    def apply_precalculated_window_c(self, x, w):
        x = _c64(x); w = np.ascontiguousarray(w, np.float32); y = np.empty_like(x)
        self.L.oracle_apply_precalculated_window_c(_p(x, _CF), _p(y, _CF), x.size, _p(w, C.c_float)); return y

    def logpower_cf(self, x, add_db=0.0):
        x = _c64(x); y = np.empty(x.size, np.float32)
        self.L.oracle_logpower_cf(_p(x, _CF), _p(y, C.c_float), x.size, add_db); return y

    def logaveragepower_cf(self, x, add_db, fft_size, avgnumber):
        """csdr.c:1663-1695: accumulate avgnumber spectra, then 10*log10 + (add_db - 10*log10(avgnumber))."""
        x = _c64(x); out = []
        adj = np.float32(np.float32(add_db) - np.float32(10.0 * np.log10(avgnumber)))
        for b in range(x.size // (fft_size * avgnumber)):
            acc = np.zeros(fft_size, np.float32)
            for n in range(avgnumber):
                seg = x[(b * avgnumber + n) * fft_size:(b * avgnumber + n + 1) * fft_size]
                self.L.oracle_accumulate_power_cf(_p(seg, _CF), _p(acc, C.c_float), fft_size)
            y = np.empty(fft_size, np.float32); self.L.oracle_log_ff(_p(acc, C.c_float), _p(y, C.c_float), fft_size, float(adj)); out.append(y)
        return np.concatenate(out) if out else np.zeros(0, np.float32)

    def shift_unroll_cc(self, x, rate, phase=0.0, size=1024):
        x = _c64(x); y = np.empty_like(x); ds = np.empty(size, np.float32); dc = np.empty(size, np.float32)
        inc = self.L.oracle_shift_unroll_init(rate, size, _p(ds, C.c_float), _p(dc, C.c_float))
        for s0 in range(0, x.size, size):
            n = min(size, x.size - s0)
            phase = self.L.oracle_shift_unroll_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, _p(ds, C.c_float), _p(dc, C.c_float), inc, phase)
        return y, float(np.float32(phase))

    def encode_ima_adpcm_i16_u8(self, x, index=0, previous=0):
        x = np.ascontiguousarray(x, np.int16); y = np.empty(x.size // 2, np.uint8); i = C.c_int(index); p = C.c_int(previous)
        self.L.oracle_encode_ima_adpcm_i16_u8(_p(x, C.c_short), _p(y, C.c_ubyte), x.size, C.byref(i), C.byref(p))
        return y, (i.value, p.value)

    def compress_fft_adpcm_f_u8(self, x, fft_size):
        """rows of fft_size dB values -> rows of (fft_size + 10) / 2 bytes"""
        x = np.ascontiguousarray(x, np.float32).reshape(-1, fft_size); y = np.empty((x.shape[0], (fft_size + 10) // 2), np.uint8)
        for r in range(x.shape[0]):
            self.L.oracle_compress_fft_adpcm_f_u8(_p(x[r], C.c_float), _p(y[r], C.c_ubyte), fft_size)
        return y

    def shift_table_init(self, size=65536):
        t = np.empty(size, np.float32); self.L.oracle_shift_table_init(_p(t, C.c_float), size); return t

    def shift_table_cc(self, x, rate, table, phase=0.0, chunk=None):
        """returns (y, phase, number of samples whose table index left the table in the reference's arithmetic)"""
        x = _c64(x); y = np.empty_like(x); table = np.ascontiguousarray(table, np.float32); chunk = chunk or max(x.size, 1); bad = 0
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0); b = C.c_int(0)
            phase = self.L.oracle_shift_table_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, rate, _p(table, C.c_float), table.size, phase, C.byref(b)); bad += b.value
        return y, float(np.float32(phase)), bad

    def shift_math_cc(self, x, rate, phase=0.0, chunk=None):
        """one call per `chunk` samples (the CLI uses its 1024-sample buffer, csdr.c:703-718); the phase chain does not depend on the cut"""
        x = _c64(x); y = np.empty_like(x); chunk = chunk or max(x.size, 1)
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0)
            phase = self.L.oracle_shift_math_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, rate, phase)
        return y, float(np.float32(phase))

    def shift_addfast_init(self, rate):
        d = np.empty(9, np.float32); self.L.oracle_shift_addfast_init(rate, _p(d, C.c_float)); return d

    def shift_addfast_cc(self, x, rate, phase=0.0, chunk=1024):
        """calls of <= chunk samples like csdr.c:781-791; samples a call leaves untouched (n % 4) come back as 0"""
        x = _c64(x); y = np.zeros_like(x); d = self.shift_addfast_init(rate); chunk = chunk or max(x.size, 1)
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0)
            phase = self.L.oracle_shift_addfast_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, _p(d, C.c_float), phase)
        return y, float(np.float32(phase))

    # ---- FFT family
    def dft(self, x, forward=True):
        x = _c64(x); y = np.empty_like(x)
        self.L.oracle_dft_c2c(_p(x, _CF), _p(y, _CF), x.size, 1 if forward else 0); return y

    def bandpass_fir_fft_cc(self, x, lo, hi, bw, window="HAMMING"):
        """Whole-stream overlap-add exactly as the CLI loop csdr.c:1833-1883 (complete blocks only)."""
        x = _c64(x)
        T = self.firdes_filter_len(bw); N = next_pow2(T)
        if N - T < 200: N <<= 1
        isz = N - T + 1; ov = T - 1
        taps = np.zeros(N, np.complex64); taps[:T] = self.firdes_bandpass_c(T, lo, hi, window)
        taps_fft = self.dft(taps)
        prev = np.zeros(N, np.complex64); out = []
        for b in range(x.size // isz):
            buf = np.zeros(N, np.complex64); buf[:isz] = x[b * isz:(b + 1) * isz]
            res = np.empty(N, np.complex64); tail = np.ascontiguousarray(prev[isz:])
            self.L.oracle_apply_fir_fft_cc(_p(buf, _CF), _p(taps_fft, _CF), _p(tail, _CF), ov, _p(res, _CF), N)
            out.append(res[:isz].copy()); prev = res
        return np.concatenate(out) if out else np.zeros(0, np.complex64)

    def fastddc_init(self, bw, decimation, shift):
        d = self._Ddc()
        err = self.L.oracle_fastddc_init(C.byref(d), bw, decimation, shift)
        return d, err

    def fastddc_geometry(self, bw, decimation, shift):
        d, _ = self.fastddc_init(bw, decimation, shift)
        return {n: getattr(d, n) for n, _t in d._fields_ if n != "dsadata"}

    def fastddc_fwd(self, x, ddc):
        """csdr.c:2288-2299: slide overlap, append input_size new samples, FFT, emit all bins (complete blocks)."""
        x = _c64(x); buf = np.zeros(ddc.fft_size, np.complex64); out = []
        for b in range(x.size // ddc.input_size):
            buf[:ddc.overlap_length] = buf[ddc.input_size:ddc.input_size + ddc.overlap_length].copy()
            buf[ddc.overlap_length:] = x[b * ddc.input_size:(b + 1) * ddc.input_size]
            out.append(self.dft(buf))
        return out

    def fastddc_inv(self, spectra, bw, decimation, shift, window="HAMMING"):
        ddc, _ = self.fastddc_init(bw, decimation, shift)
        tf = np.empty(ddc.fft_size, np.complex64)
        self.L.oracle_fastddc_make_taps_fft(C.byref(ddc), shift, decimation, WINDOWS[window], _p(tf, _CF))
        st = _DShiftStatus(0, 0.0, 0); out = []
        for sp in spectra:
            sp = _c64(sp); y = np.empty(ddc.post_input_size, np.complex64)
            st = self.L.oracle_fastddc_inv_cc(_p(sp, _CF), _p(y, _CF), C.byref(ddc), _p(tf, _CF), st)
            out.append(y[:st.output_size].copy())
        return np.concatenate(out) if out else np.zeros(0, np.complex64)


def next_pow2(x: int) -> int:
    for b in range(31):
        if x < (1 << b):
            return 1 << b
    return -1


def _stream_fracdec(call, d, x, block):
    """Drive a fractional decimator over ``x``.  block=None: one call on the whole array.
    Otherwise reproduce the CLI's re-feeding of the unconsumed tail (csdr.c:1510-1522), complete reads only."""
    if block is None:
        out = np.empty(int(x.size / max(d.rate, 1.0)) + 16, np.float32)
        call(x, out, x.size)
        return out[:d.output_size].copy()
    buf = np.zeros(block, np.float32); outs = []; pos = 0
    out = np.empty(block, np.float32)
    while True:
        if d.input_processed == 0:
            need = block; keep = 0
        else:
            need = d.input_processed; keep = block - need
            buf[:keep] = buf[need:].copy()
        if pos + need > x.size:
            break
        buf[keep:] = x[pos:pos + need]; pos += need
        if d.input_processed == 0:
            d.input_processed = block
        call(buf, out, block)
        outs.append(out[:d.output_size].copy())
    return np.concatenate(outs) if outs else np.zeros(0, np.float32)


# ======================================================================================================
class Ref:
    """Binding of the compiled, unmodified reference library (libcsdr.h / libcsdr_gpl.h / fastddc.h ABI)."""

    name = "reference"

    class _FracDec(C.Structure):            # libcsdr.h:151-168
        _fields_ = [("where", C.c_float), ("input_processed", C.c_int), ("output_size", C.c_int),
                    ("num_poly_points", C.c_int), ("poly_precalc_denomiator", C.POINTER(C.c_float)),
                    ("coeffs_buf", C.POINTER(C.c_float)), ("filtered_buf", C.POINTER(C.c_float)),
                    ("xifirst", C.c_int), ("xilast", C.c_int), ("rate", C.c_float),
                    ("taps", C.POINTER(C.c_float)), ("taps_length", C.c_int)]

    class _Agc(C.Structure):                # libcsdr.h:118-128
        _fields_ = [("buffer_1", C.POINTER(C.c_float)), ("buffer_2", C.POINTER(C.c_float)),
                    ("buffer_input", C.POINTER(C.c_float)), ("peak_1", C.c_float), ("peak_2", C.c_float),
                    ("input_size", C.c_int), ("reference", C.c_float), ("last_gain", C.c_float)]

    class _Unroll(C.Structure):             # libcsdr.h:199-205
        _fields_ = [("dsin", C.POINTER(C.c_float)), ("dcos", C.POINTER(C.c_float)), ("phase_increment", C.c_float), ("size", C.c_int)]

    class _Table(C.Structure):              # libcsdr.h:180-184
        _fields_ = [("table", C.POINTER(C.c_float)), ("table_size", C.c_int)]

    class _Ima(C.Structure):                # ima_adpcm.h:35-38
        _fields_ = [("index", C.c_int), ("previousValue", C.c_int)]

    class _AddFast(C.Structure):            # libcsdr.h:189-194
        _fields_ = [("dsin", C.c_float * 4), ("dcos", C.c_float * 4), ("phase_increment", C.c_float)]

    class _Plan(C.Structure):               # fft_fftw.h:14-20
        _fields_ = [("size", C.c_int), ("input", C.c_void_p), ("output", C.c_void_p), ("plan", C.c_void_p)]

    class _Ddc(C.Structure):                # fastddc.h:5-24
        _fields_ = [(n, C.c_int) for n in ("pre_decimation", "post_decimation", "taps_length", "taps_min_length",
                                           "overlap_length", "fft_size", "fft_inv_size", "input_size",
                                           "post_input_size")] + \
                   [("pre_shift", C.c_float), ("startbin", C.c_int), ("v", C.c_int), ("offsetbin", C.c_int),
                    ("post_shift", C.c_float), ("output_scrape", C.c_int), ("scrap", C.c_int), ("dsadata", _Shift)]

    def __init__(self, path: Path = REF_SO):
        if not path.exists():
            raise FileNotFoundError(f"{path} missing: run `make -C oracle ref` where /root/reference exists")
        L = self.L = C.CDLL(str(path))
        L.firdes_filter_len.argtypes = [C.c_float]
        L.firdes_lowpass_f.argtypes = [C.POINTER(C.c_float), C.c_int, C.c_float, C.c_int]
        L.firdes_bandpass_c.argtypes = [C.POINTER(_CF), C.c_int, C.c_float, C.c_float, C.c_int]
        L.shift_addition_init.argtypes = [C.c_float]; L.shift_addition_init.restype = _Shift
        L.shift_addition_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, _Shift, C.c_float]
        L.shift_addition_cc.restype = C.c_float
        L.decimating_shift_addition_init.argtypes = [C.c_float, C.c_int]; L.decimating_shift_addition_init.restype = _Shift
        L.decimating_shift_addition_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, _Shift, C.c_int, _DShiftStatus]
        L.decimating_shift_addition_cc.restype = _DShiftStatus
        L.fir_decimate_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_int, C.POINTER(C.c_float), C.c_int]
        L.fmdemod_quadri_cf.argtypes = [C.POINTER(_CF), C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_float), _CF]
        L.fmdemod_quadri_cf.restype = _CF
        L.fractional_decimator_ff_init.argtypes = [C.c_float, C.c_int, C.POINTER(C.c_float), C.c_int]
        L.fractional_decimator_ff_init.restype = self._FracDec
        L.fractional_decimator_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.POINTER(self._FracDec)]
        L.fastagc_ff.argtypes = [C.POINTER(self._Agc), C.POINTER(C.c_float)]
        L.deemphasis_wfm_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_float, C.c_int, C.c_float]
        L.deemphasis_wfm_ff.restype = C.c_float
        L.limit_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_float]
        L.deemphasis_nfm_ff.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_int]
        fp = C.POINTER(C.c_float)
        L.precalculate_window.argtypes = [C.c_int, C.c_int]; L.precalculate_window.restype = fp
        L.apply_precalculated_window_c.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, fp]
        L.logpower_cf.argtypes = [C.POINTER(_CF), fp, C.c_int, C.c_float]
        L.accumulate_power_cf.argtypes = [C.POINTER(_CF), fp, C.c_int]
        L.log_ff.argtypes = [fp, fp, C.c_int, C.c_float]
        L.shift_unroll_init.argtypes = [C.c_float, C.c_int]; L.shift_unroll_init.restype = self._Unroll
        L.shift_unroll_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.POINTER(self._Unroll), C.c_float]; L.shift_unroll_cc.restype = C.c_float
        L.shift_math_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_float, C.c_float]; L.shift_math_cc.restype = C.c_float
        L.shift_table_init.argtypes = [C.c_int]; L.shift_table_init.restype = self._Table
        L.shift_table_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.c_float, self._Table, C.c_float]; L.shift_table_cc.restype = C.c_float
        L.encode_ima_adpcm_i16_u8.argtypes = [C.POINTER(C.c_short), C.POINTER(C.c_ubyte), C.c_int, self._Ima]; L.encode_ima_adpcm_i16_u8.restype = self._Ima
        L.shift_addfast_init.argtypes = [C.c_float]; L.shift_addfast_init.restype = self._AddFast
        L.shift_addfast_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.c_int, C.POINTER(self._AddFast), C.c_float]; L.shift_addfast_cc.restype = C.c_float
        L.make_fft_c2c.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int]; L.make_fft_c2c.restype = C.POINTER(self._Plan)
        L.fft_execute.argtypes = [C.POINTER(self._Plan)]
        L.fft_destroy.argtypes = [C.POINTER(self._Plan)]
        L.apply_fir_fft_cc.argtypes = [C.POINTER(self._Plan), C.POINTER(self._Plan), C.POINTER(_CF), C.POINTER(_CF), C.c_int]
        L.fastddc_init.argtypes = [C.POINTER(self._Ddc), C.c_float, C.c_int, C.c_float]
        L.fft_swap_sides.argtypes = [C.POINTER(_CF), C.c_int]
        L.fastddc_inv_cc.argtypes = [C.POINTER(_CF), C.POINTER(_CF), C.POINTER(self._Ddc), C.POINTER(self._Plan), C.POINTER(_CF), _DShiftStatus]
        L.fastddc_inv_cc.restype = _DShiftStatus
        L.next_pow2.argtypes = [C.c_int]

    def convert_u8_f(self, x):
        x = np.ascontiguousarray(x, np.uint8); y = np.empty(x.size, np.float32)
        self.L.convert_u8_f(_p(x, C.c_ubyte), _p(y, C.c_float), x.size); return y

    def convert_s16_f(self, x):
        x = np.ascontiguousarray(x, np.int16); y = np.empty(x.size, np.float32)
        self.L.convert_s16_f(_p(x, C.c_short), _p(y, C.c_float), x.size); return y

    def convert_f_s16(self, x):
        x = np.ascontiguousarray(x, np.float32); y = np.empty(x.size, np.int16)
        self.L.convert_f_s16(_p(x, C.c_float), _p(y, C.c_short), x.size); return y

    def firdes_filter_len(self, bw): return int(self.L.firdes_filter_len(bw))

    def firdes_lowpass_f(self, length, cutoff, window="HAMMING"):
        t = np.empty(length, np.float32)
        self.L.firdes_lowpass_f(_p(t, C.c_float), length, cutoff, WINDOWS[window]); return t

    def firdes_bandpass_c(self, length, lo, hi, window="HAMMING"):
        t = np.empty(length, np.complex64)
        self.L.firdes_bandpass_c(_p(t, _CF), length, lo, hi, WINDOWS[window]); return t

    def shift_addition_init(self, rate):
        d = self.L.shift_addition_init(rate); return (d.sindelta, d.cosdelta, d.rate)

    def shift_addition_cc(self, x, rate, phase=0.0, chunk=None):
        x = _c64(x); y = np.empty_like(x); d = self.L.shift_addition_init(rate)
        chunk = chunk or max(x.size, 1)
        for s in range(0, x.size, chunk):
            n = min(chunk, x.size - s)
            phase = self.L.shift_addition_cc(_p(x[s:], _CF), _p(y[s:], _CF), n, d, phase)
        return y, float(np.float32(phase))

    def decimating_shift_addition_cc(self, x, rate, decimation, remain=0, phase=0.0):
        x = _c64(x); y = np.empty(x.size // decimation + 2, np.complex64)
        d = self.L.decimating_shift_addition_init(rate, decimation)
        st = self.L.decimating_shift_addition_cc(_p(x, _CF), _p(y, _CF), x.size, d, decimation, _DShiftStatus(remain, phase, 0))
        return y[:st.output_size].copy(), (st.decimation_remain, st.starting_phase)

    def fir_decimate_cc(self, x, decimation, taps):
        x = _c64(x); taps = np.ascontiguousarray(taps, np.float32)
        y = np.empty(max(x.size // decimation + 1, 1), np.complex64)
        n = self.L.fir_decimate_cc(_p(x, _CF), _p(y, _CF), x.size, decimation, _p(taps, C.c_float), taps.size)
        return y[:n].copy()

    def fmdemod_quadri_cf(self, x, last=0j):
        x = _c64(x); y = np.empty(x.size, np.float32); tmp = np.empty(2 * x.size + 4, np.float32)
        r = self.L.fmdemod_quadri_cf(_p(x, _CF), _p(y, C.c_float), x.size, _p(tmp, C.c_float),
                                     _CF(np.float32(last.real), np.float32(last.imag)))
        return y, complex(r.i, r.q)

    def fractional_decimator_ff(self, x, rate, num_poly_points=12, taps=None, block=None):
        x = np.ascontiguousarray(x, np.float32)
        tp = np.ascontiguousarray(taps, np.float32) if taps is not None else None
        self._keep = tp
        d = self.L.fractional_decimator_ff_init(rate, num_poly_points, _p(tp, C.c_float) if tp is not None else None,
                                                tp.size if tp is not None else 0)
        return _stream_fracdec(lambda buf, out, n: self.L.fractional_decimator_ff(_p(buf, C.c_float), _p(out, C.c_float), n, C.byref(d)),
                               d, x, block)

    def fastagc_ff(self, x, block=1024, reference=1.0):
        x = np.ascontiguousarray(x, np.float32); nblk = x.size // block
        bufs = [np.zeros(block, np.float32) for _ in range(3)]
        byaddr = {b.ctypes.data: b for b in bufs}
        st = self._Agc(_p(bufs[0], C.c_float), _p(bufs[1], C.c_float), _p(bufs[2], C.c_float), 0, 0, block, reference, 0)
        y = np.empty(nblk * block, np.float32)
        for b in range(nblk):
            byaddr[C.cast(st.buffer_input, C.c_void_p).value][:] = x[b * block:(b + 1) * block]
            self.L.fastagc_ff(C.byref(st), _p(y[b * block:], C.c_float))
        return y

    def deemphasis_wfm_ff(self, x, tau, sample_rate, last=0.0, block=None):
        x = np.ascontiguousarray(x, np.float32); y = np.empty_like(x); block = block or max(x.size, 1)
        for s0 in range(0, x.size, block):
            n = min(block, x.size - s0)
            last = self.L.deemphasis_wfm_ff(_p(x[s0:], C.c_float), _p(y[s0:], C.c_float), n, tau, sample_rate, last)
        return y, float(np.float32(last))

    def limit_ff(self, x, max_amplitude=1.0):
        x = np.ascontiguousarray(x, np.float32); y = np.empty_like(x)
        self.L.limit_ff(_p(x, C.c_float), _p(y, C.c_float), x.size, max_amplitude); return y

    NFM_RATES = (48000, 44100, 11025, 8000)

    def deemphasis_nfm_ff(self, x, sample_rate):
        x = np.ascontiguousarray(x, np.float32); y = np.zeros_like(x)
        n = self.L.deemphasis_nfm_ff(_p(x, C.c_float), _p(y, C.c_float), x.size, sample_rate)
        return y[:n].copy()

    def deemphasis_nfm_taps(self, sample_rate):
        """the table the compiled reference exports for this rate (length from the ELF symbol size)"""
        import re, subprocess
        for line in subprocess.check_output(["nm", "-S", "--defined-only", self.L._name], text=True).splitlines():
            m = re.match(r"^[0-9a-f]+ ([0-9a-f]+) D deemphasis_nfm_predefined_fir_%d$" % sample_rate, line)
            if m:
                n = int(m.group(1), 16) // 4
                return np.array((C.c_float * n).in_dll(self.L, "deemphasis_nfm_predefined_fir_%d" % sample_rate), np.float32)
        return None

    def precalculate_window(self, size, window="HAMMING"):
        p = self.L.precalculate_window(size, WINDOWS[window]); return np.ctypeslib.as_array(p, shape=(size,)).copy()

    def apply_precalculated_window_c(self, x, w):
        x = _c64(x); w = np.ascontiguousarray(w, np.float32); y = np.empty_like(x)
        self.L.apply_precalculated_window_c(_p(x, _CF), _p(y, _CF), x.size, _p(w, C.c_float)); return y

    def logpower_cf(self, x, add_db=0.0):
        x = _c64(x); y = np.empty(x.size, np.float32)
        self.L.logpower_cf(_p(x, _CF), _p(y, C.c_float), x.size, add_db); return y

    def logaveragepower_cf(self, x, add_db, fft_size, avgnumber):
        x = _c64(x); out = []
        adj = np.float32(np.float32(add_db) - np.float32(10.0 * np.log10(avgnumber)))
        for b in range(x.size // (fft_size * avgnumber)):
            acc = np.zeros(fft_size, np.float32)
            for n in range(avgnumber):
                seg = x[(b * avgnumber + n) * fft_size:(b * avgnumber + n + 1) * fft_size]
                self.L.accumulate_power_cf(_p(seg, _CF), _p(acc, C.c_float), fft_size)
            y = np.empty(fft_size, np.float32); self.L.log_ff(_p(acc, C.c_float), _p(y, C.c_float), fft_size, float(adj)); out.append(y)
        return np.concatenate(out) if out else np.zeros(0, np.float32)

    def shift_unroll_cc(self, x, rate, phase=0.0, size=1024):
        x = _c64(x); y = np.empty_like(x)
        d = self.L.shift_unroll_init(rate, size)
        for s0 in range(0, x.size, size):
            n = min(size, x.size - s0)
            phase = self.L.shift_unroll_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, C.byref(d), phase)
        return y, float(np.float32(phase))

    def shift_table_init(self, size=65536):
        d = self.L.shift_table_init(size); return np.ctypeslib.as_array(d.table, shape=(size,)).copy()

    def shift_table_cc(self, x, rate, table, phase=0.0, chunk=None):
        x = _c64(x); y = np.empty_like(x); table = np.ascontiguousarray(table, np.float32); chunk = chunk or max(x.size, 1)
        d = self._Table(_p(table, C.c_float), table.size)
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0)
            phase = self.L.shift_table_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, rate, d, phase)
        return y, float(np.float32(phase))

    def encode_ima_adpcm_i16_u8(self, x, index=0, previous=0):
        x = np.ascontiguousarray(x, np.int16); y = np.empty(x.size // 2, np.uint8)
        st = self.L.encode_ima_adpcm_i16_u8(_p(x, C.c_short), _p(y, C.c_ubyte), x.size, self._Ima(index, previous))
        return y, (st.index, st.previousValue)

    def shift_math_cc(self, x, rate, phase=0.0, chunk=None):
        x = _c64(x); y = np.empty_like(x); chunk = chunk or max(x.size, 1)
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0)
            phase = self.L.shift_math_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, rate, phase)
        return y, float(np.float32(phase))

    def shift_addfast_init(self, rate):
        d = self.L.shift_addfast_init(rate); return np.array(list(d.dsin) + list(d.dcos) + [d.phase_increment], np.float32)

    def shift_addfast_cc(self, x, rate, phase=0.0, chunk=1024):
        x = _c64(x); y = np.zeros_like(x); d = self.L.shift_addfast_init(rate); chunk = chunk or max(x.size, 1)
        for s0 in range(0, x.size, chunk):
            n = min(chunk, x.size - s0)
            phase = self.L.shift_addfast_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), n, C.byref(d), phase)
        return y, float(np.float32(phase))

    def dft(self, x, forward=True):
        x = _c64(x).copy(); y = np.empty_like(x)
        pl = self.L.make_fft_c2c(x.size, x.ctypes.data, y.ctypes.data, 1 if forward else 0, 0)
        self.L.fft_execute(pl); self.L.fft_destroy(pl); return y

    def bandpass_fir_fft_cc(self, x, lo, hi, bw, window="HAMMING"):
        x = _c64(x)
        T = self.firdes_filter_len(bw); N = int(self.L.next_pow2(T))
        if N - T < 200: N <<= 1
        isz = N - T + 1; ov = T - 1
        taps = np.zeros(N, np.complex64); taps[:T] = self.firdes_bandpass_c(T, lo, hi, window)
        taps_fft = self.dft(taps)
        inp = np.zeros(N, np.complex64); spec = np.empty(N, np.complex64); ospec = np.empty(N, np.complex64)
        o = [np.zeros(N, np.complex64), np.zeros(N, np.complex64)]
        pf = self.L.make_fft_c2c(N, inp.ctypes.data, spec.ctypes.data, 1, 0)
        pi = [self.L.make_fft_c2c(N, ospec.ctypes.data, o[k].ctypes.data, 0, 0) for k in range(2)]
        out = []
        for b in range(x.size // isz):
            inp[:isz] = x[b * isz:(b + 1) * isz]
            cur, prev = (1, 0) if b & 1 else (0, 1)
            tail = o[prev][isz:]
            self.L.apply_fir_fft_cc(pf, pi[cur], _p(taps_fft, _CF), C.cast(tail.ctypes.data, C.POINTER(_CF)), ov)
            out.append(o[cur][:isz].copy())
        self.L.fft_destroy(pf); [self.L.fft_destroy(p) for p in pi]
        return np.concatenate(out) if out else np.zeros(0, np.complex64)

    def fastddc_init(self, bw, decimation, shift):
        d = self._Ddc()
        err = self.L.fastddc_init(C.byref(d), bw, decimation, shift)
        return d, err

    def fastddc_geometry(self, bw, decimation, shift):
        d, _ = self.fastddc_init(bw, decimation, shift)
        return {n: getattr(d, n) for n, _t in d._fields_ if n not in ("dsadata", "output_scrape")}

    def fastddc_fwd(self, x, ddc):
        x = _c64(x); buf = np.zeros(ddc.fft_size, np.complex64); out = []
        for b in range(x.size // ddc.input_size):
            buf[:ddc.overlap_length] = buf[ddc.input_size:ddc.input_size + ddc.overlap_length].copy()
            buf[ddc.overlap_length:] = x[b * ddc.input_size:(b + 1) * ddc.input_size]
            out.append(self.dft(buf))
        return out

    def fastddc_inv(self, spectra, bw, decimation, shift, window="HAMMING"):
        ddc, _ = self.fastddc_init(bw, decimation, shift)
        taps = np.zeros(ddc.fft_size, np.complex64)
        hb = np.float32(0.5 / decimation); sh = np.float32(shift)
        taps[:ddc.taps_length] = self.firdes_bandpass_c(ddc.taps_length, float(-sh - hb), float(-sh + hb), window)
        tf = self.dft(taps); self.L.fft_swap_sides(_p(tf, _CF), ddc.fft_size)
        ii = np.zeros(ddc.fft_inv_size, np.complex64); io = np.zeros(ddc.fft_inv_size, np.complex64)
        pl = self.L.make_fft_c2c(ddc.fft_inv_size, ii.ctypes.data, io.ctypes.data, 0, 0)
        st = _DShiftStatus(0, 0.0, 0); out = []
        for sp in spectra:
            sp = _c64(sp).copy(); y = np.empty(ddc.post_input_size, np.complex64)
            st = self.L.fastddc_inv_cc(_p(sp, _CF), _p(y, _CF), C.byref(ddc), pl, _p(tf, _CF), st)
            out.append(y[:st.output_size].copy())
        self.L.fft_destroy(pl)
        return np.concatenate(out) if out else np.zeros(0, np.complex64)


def have_ref() -> bool:
    return REF_SO.exists()


def pick_idx(n: int, k: int) -> np.ndarray:
    """the k seeded positions of an n-sample output at which tests/golden stores the reference's values (a function of n and k alone)"""
    return np.sort(np.random.default_rng(n).choice(n, min(k, n), replace=False))


def rel_rms(y, ref) -> float:
    """sqrt(sum|y-ref|^2 / sum|ref|^2) -- the parity metric of SURVEY.md section 8(d)."""
    y = np.asarray(y); ref = np.asarray(ref)
    den = float(np.sum(np.abs(ref.astype(np.complex128)) ** 2))
    num = float(np.sum(np.abs(y.astype(np.complex128) - ref.astype(np.complex128)) ** 2))
    return (num / den) ** 0.5 if den > 0 else (0.0 if num == 0 else float("inf"))
