#!/usr/bin/env python
"""Regenerate tests/golden/ref_outputs.npz: what the compiled, unmodified reference (oracle/_ref, `make -C oracle ref REF=<csdr tree>`)
computes on the seeded inputs of the tests that compare the product or the oracle with it, so those tests run without the reference.

Long outputs are stored at seeded positions derived from their length (oracle.pyoracle.pick_idx): key + "_n" is the length, key the
values; the tests compare their own output at the same positions.
Outputs the tests require to be bit-identical are stored as the SHA-256 of their bytes (key + "_sha").
Inputs are rebuilt here exactly as the tests build them (numpy's PCG64 streams are stable across versions).

    python tests/golden/make_ref_outputs.py
"""
from pathlib import Path
import hashlib
import sys

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle.pyoracle import Ref, pick_idx  # noqa: E402

OUT = Path(__file__).resolve().parent / "ref_outputs.npz"
SAMPLE, CPU_SAMPLE = 1024, 256        # positions kept of a long output: GPU tests, CPU oracle tests


def cplx(rng, n, amp=1.0):
    return ((rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)) * amp).astype(np.complex64)


def pick(g, key, y, k=SAMPLE):
    g[key + "_n"] = np.int64(y.size)
    g[key] = y[pick_idx(y.size, k)]


def sha(a) -> np.ndarray:
    return np.array(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


def main():
    r = Ref(); g = {}
    # test_gpu_parity.py::test_fir_golden_and_reference
    x = cplx(np.random.default_rng(5), 262144)
    g["fir_taps_199_0p05"] = taps = r.firdes_lowpass_f(199, 0.05)
    pick(g, "fir_262144_d10", r.fir_decimate_cc(x, 10, taps))
    # test_gpu_parity2.py::test_shift_dropin_and_golden: one 65536-step chain (the drift grows along it: sample it all the way)
    x = cplx(np.random.default_rng(3), 1 << 16)
    y, ph = r.shift_addition_cc(x, -0.3, 0.0, None)
    pick(g, "shift_65536_m0p3", y); g["shift_65536_m0p3_phase"] = np.float32(ph)
    # test_gpu_parity2.py::test_bandpass_fir_fft_dropin_golden_and_reference: BASELINE config 5 geometry
    x = cplx(np.random.default_rng(6), 2098 * 5)
    pick(g, "bandpass_cfg5", r.bandpass_fir_fft_cc(x, -0.05, 0.05, 0.002))
    # test_gpu_parity2.py::test_fastddc_config3_bank_vs_oracle_and_reference: 896 outputs, stored whole
    bw, dec, nblocks, n = 0.002, 64, 4, 4 * 14336
    rng = np.random.default_rng(8)
    shifts = [-0.4, -0.2113, 0.0, 0.1, 0.3337]
    t = np.arange(n)
    x = sum(np.exp(2j * np.pi * (s + 0.001) * t) for s in shifts).astype(np.complex64) / len(shifts) + cplx(rng, n, 0.05)
    rd, _ = r.fastddc_init(bw, dec, 0.1)
    g["fastddc_cfg3_shift0p1"] = r.fastddc_inv(r.fastddc_fwd(x, rd), bw, dec, 0.1)
    # test_gpu_round2.py::test_config2_against_compiled_reference_8x262144
    taps = r.firdes_lowpass_f(199, 0.5 / 10)
    for c in range(8):
        x = cplx(np.random.default_rng(100 + c), 262_144)
        pick(g, f"cfg2_ch{c}", r.fir_decimate_cc(x, 10, taps), 512)
    cpu_tests(r, g)
    cpu_tests_2(r, g)
    np.savez_compressed(OUT, **g)
    print(f"{OUT}: {OUT.stat().st_size} bytes, {len(g)} arrays")


def cpu_tests(r, g):
    """tests/test_oracle.py: the oracle restatement against the reference build"""
    # test_ref_audio_tail
    x = np.random.default_rng(21).uniform(-2, 2, 1 << 16).astype(np.float32)
    x[7] = np.nan; x[9] = np.inf; x[11] = -np.inf
    g["limit_0p7_sha"] = sha(r.limit_ff(x, 0.7))
    x = np.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)
    for i, (tau, fs, last, blk) in enumerate(((50e-6, 48000, 0.0, 1024), (75e-6, 240000, float("nan"), None), (50e-6, 44100, 0.3, 4096))):
        y, l = r.deemphasis_wfm_ff(x, tau, fs, last, blk)
        g[f"deemph_wfm_{i}_sha"] = sha(y); g[f"deemph_wfm_{i}_last"] = np.float32(l)
    # test_ref_nco_deltas_over_many_rates
    rng = np.random.default_rng(0)
    rates = np.concatenate([rng.uniform(-0.5, 0.5, 6000), rng.uniform(-5, 5, 500), [0, 0.25, -0.25, 0.5, -0.5, 1e-7, -1e-7]]).astype(np.float32)
    g["nco_deltas_sha"] = sha(np.array([r.shift_addition_init(float(v)) for v in rates], np.float32))
    # test_ref_conversions_all_codes
    g["conv_u8_sha"] = sha(r.convert_u8_f(np.arange(256, dtype=np.uint8)))
    g["conv_s16_sha"] = sha(r.convert_s16_f(np.arange(-32768, 32768).astype(np.int16)))
    g["conv_f_s16_sha"] = sha(r.convert_f_s16(np.random.default_rng(3).uniform(-1, 1, 1 << 18).astype(np.float32)))
    # test_ref_fir_decimate
    for T, D, bw in ((79, 10, 0.05), (199, 10, 0.0201), (801, 50, 0.005)):
        g[f"firdes_len_{T}"] = np.int64(r.firdes_filter_len(bw))
        g[f"firdes_taps_{T}"] = taps = r.firdes_lowpass_f(T, 0.5 / D)
        x = cplx(np.random.default_rng(T), 262144)
        pick(g, f"fir_dec_{T}", r.fir_decimate_cc(x, D, taps), CPU_SAMPLE)
    # test_ref_shift_addition
    x = cplx(np.random.default_rng(7), 1 << 17)
    for i, (rate, chunk) in enumerate(((-0.085, 1024), (0.2, 1024), (0.4999, 1024), (0.01, 16384), (-0.3, None))):
        y, ph = r.shift_addition_cc(x, rate, 0.0, chunk)
        pick(g, f"shift_add_{i}", y, CPU_SAMPLE); g[f"shift_add_{i}_phase"] = np.float32(ph)
    # test_ref_fmdemod_fracdec_agc
    rng = np.random.default_rng(11)
    t = np.arange(1 << 16)
    fm = np.exp(1j * np.cumsum(0.4 * np.sin(2 * np.pi * t / 300))).astype(np.complex64)
    y, last = r.fmdemod_quadri_cf(fm)
    g["fmdemod_sha"] = sha(y); g["fmdemod_last"] = np.complex64(last)
    aud = rng.uniform(-1, 1, 1 << 16).astype(np.float32)
    for i, (rate, blk) in enumerate(((5.0, 1024), (5.0, None), (1.5, 1024), (48.0 / 44.1, 4096))):
        pick(g, f"fracdec_{i}", r.fractional_decimator_ff(aud, rate, 12, None, blk), CPU_SAMPLE)
    for i, (block, refl) in enumerate(((1024, 1.0), (100, 0.3))):
        pick(g, f"agc_{i}", r.fastagc_ff(aud * 0.05, block, refl), CPU_SAMPLE)


def cpu_tests_2(r, g):
    """tests/test_oracle.py, continued: samples without stored positions (pick_idx), the shift tables as their differences from the oracle's"""
    from oracle.pyoracle import Oracle
    o = Oracle()
    # test_golden_and_ref_deemphasis_nfm
    x = np.random.default_rng(4).uniform(-1, 1, 20_000).astype(np.float32)
    for rate in r.NFM_RATES:
        pick(g, f"nfm_{rate}", r.deemphasis_nfm_ff(x, rate), 256)
    g["nfm_22050_n"] = np.int64(r.deemphasis_nfm_ff(x, 22050).size)
    # test_golden_and_ref_shift_addfast
    z = (np.random.default_rng(8).standard_normal(20_000) + 1j * np.random.default_rng(9).standard_normal(20_000)).astype(np.complex64)
    for rate in (0.25, 0.125):
        g[f"addfast_init_{rate}"] = r.shift_addfast_init(rate)
        for chunk in (1024, 4096, None):
            y, ph = r.shift_addfast_cc(z, rate, 0.3, chunk)
            pick(g, f"addfast_{rate}_{chunk}", y, 128); g[f"addfast_{rate}_{chunk}_phase"] = np.float32(ph)
    y, ph = r.shift_addfast_cc(z, 0.25, -1.0, 1022)
    pick(g, "addfast_1022", y, 128); g["addfast_1022_phase"] = np.float32(ph); g["addfast_1022_tail"] = y[1020:1022]
    # test_ref_shift_table_bit_exact: the oracle's output on the reference's own tables, all (rate, phase) cases in one digest per size
    x = (np.random.default_rng(1).standard_normal(60_000) + 1j * np.random.default_rng(2).standard_normal(60_000)).astype(np.complex64)
    for size in (65536, 1024, 100):
        t = r.shift_table_init(size); mine = o.shift_table_init(size)
        ulps = t.view(np.int32).astype(np.int64) - mine.view(np.int32)          # a one-ulp step here and there (the build's libmvec sin)
        assert np.abs(ulps).max() <= 127
        g[f"table_{size}_ulps"] = ulps.astype(np.int8)
        outs = []
        for rate in (-0.5, -0.31, -0.085, 0.0, 1e-4, 0.2, 0.25, 0.4999, 0.5):
            for ph0 in (0.0, 3.0, 1.5707964, 6.2831855):
                b, pb = r.shift_table_cc(x, rate, t, ph0)
                outs += [b.tobytes(), np.float32(pb).tobytes()]
        g[f"table_{size}_sha"] = np.array(hashlib.sha256(b"".join(outs)).hexdigest())
    # test_golden_and_ref_shift_math
    z = (np.random.default_rng(8).standard_normal(30_000) + 1j * np.random.default_rng(9).standard_normal(30_000)).astype(np.complex64)
    for i, rate in enumerate((-0.5, -0.31, 0.0, 1e-4, 0.2, 0.4999, 0.5)):
        for j, (ph0, chunk) in enumerate(((0.0, 1024), (3.0, None), (-7.5, 1000), (100.0, 1024))):
            y, ph = r.shift_math_cc(z, rate, ph0, chunk)
            pick(g, f"math_{i}_{j}", y, 64); g[f"math_{i}_{j}_phase"] = np.float32(ph)
    # test_ref_ima_adpcm: encoder bytes and state, and the reference CLI's compressed waterfall lines
    rng = np.random.default_rng(0)
    for n in (2, 10, 1000, 4097):
        x = (rng.standard_normal(n) * rng.choice([10, 300, 5000, 40000])).clip(-32768, 32767).astype(np.int16)
        b, st = r.encode_ima_adpcm_i16_u8(x, 3, -200)
        g[f"ima_{n}_sha"] = sha(b); g[f"ima_{n}_state"] = np.array(st, np.int64)
    import subprocess
    from oracle.pyoracle import REF_CLI
    db = rng.uniform(-120, -20, (5, 512)).astype(np.float32)
    p = subprocess.run([str(REF_CLI), "compress_fft_adpcm_f_u8", "512"], input=db.tobytes(), stdout=subprocess.PIPE, check=True, timeout=60)
    g["adpcm_lines_512"] = np.frombuffer(p.stdout, np.uint8)[:5 * (512 + 10) // 2]
    # test_ref_fft_paths
    rng = np.random.default_rng(13)
    x = cplx(rng, 2098 * 4)
    pick(g, "fft_bandpass", r.bandpass_fir_fft_cc(x, -0.05, 0.05, 0.002), 256)
    ddc, _ = o.fastddc_init(0.002, 64, -0.2)
    xs = cplx(rng, ddc.input_size * 2)
    rd, _ = r.fastddc_init(0.002, 64, -0.2)
    sb = r.fastddc_fwd(xs, rd)
    pick(g, "fft_ddc_fwd", np.stack(sb).reshape(-1), 512)
    g["fft_ddc_inv"] = r.fastddc_inv(sb, 0.002, 64, -0.2)


if __name__ == "__main__":
    main()
