"""CPU tests: the oracle restatement (oracle/oracle.c) against
  (1) the committed golden vectors produced by the compiled reference (tests/golden/make_golden.py), and
  (2) the compiled reference on larger seeded inputs: its outputs stored by tests/golden/make_ref_outputs.py (digests of the
      outputs required bit-exact, seeded samples of the others), or the library itself (oracle/_ref) when it is built.

Tolerances: bit-exact where the reference build performs the same IEEE operations (conversions, NCO
recursion, fmdemod, fractional decimator, fastagc, geometry); <= 1e-6 relative RMS where the
reference's -ffast-math build may re-associate sums or swap libm calls (FIR sums, tap design, FFT).
The north-star tolerance for float blocks is 1e-5 relative RMS.
"""
import hashlib
from pathlib import Path

import numpy as np
import pytest

from oracle.pyoracle import have_ref, pick_idx, rel_rms

GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_golden.npz")
REF = np.load(Path(__file__).parent / "golden" / "ref_outputs.npz")
TIGHT = 1e-6


# ------------------------------------------------------------------ golden vectors
def test_golden_conversions_bit_exact(oracle):
    assert np.array_equal(oracle.convert_u8_f(GOLD["u8_in"]), GOLD["u8_out"])
    assert np.array_equal(oracle.convert_s16_f(GOLD["s16_in"]), GOLD["s16_out"])
    assert np.array_equal(oracle.convert_f_s16(GOLD["f_in"]), GOLD["f_s16_out"])
    # the known answers SURVEY 8(a) quotes
    t = oracle.convert_u8_f(np.array([0, 127, 128, 255], np.uint8))
    assert t[0] == -1.0 and t[3] == 1.0 and t[1] == np.float32(-0.00392156886) and t[2] == np.float32(0.00392156886)
    assert list(oracle.convert_f_s16(np.array([-1, 0.25, 1.5, 2.0], np.float32))) == [-32767, 8191, -16386, -2]


def test_golden_filter_design(oracle):
    lens = [oracle.firdes_filter_len(float(b)) for b in GOLD["filter_len_bw"]]
    assert lens == list(GOLD["filter_len"])
    assert lens[:5] == [79, 199, 201, 801, 1999]
    assert rel_rms(oracle.firdes_lowpass_f(79, 0.05), GOLD["lowpass_79"]) < TIGHT
    assert rel_rms(oracle.firdes_lowpass_f(199, 0.05), GOLD["lowpass_199"]) < TIGHT
    assert rel_rms(oracle.firdes_lowpass_f(101, 0.1, "BLACKMAN"), GOLD["lowpass_101_blackman"]) < TIGHT
    assert rel_rms(oracle.firdes_bandpass_c(79, 0.1, 0.3), GOLD["bandpass_79"]) < TIGHT
    t = oracle.firdes_lowpass_f(199, 0.05)
    assert np.array_equal(t, t[::-1]) and abs(float(t.sum()) - 1.0) < 1e-6


def test_golden_shift(oracle):
    y, ph = oracle.shift_addition_cc(GOLD["shift_in"], -0.085, 0.0, 1024)
    assert rel_rms(y, GOLD["shift_out_chunk1024"]) < 1e-7 and np.float32(ph) == GOLD["shift_phase_chunk1024"]
    y, ph = oracle.shift_addition_cc(GOLD["shift_in"], 0.2, 0.3, None)
    assert rel_rms(y, GOLD["shift_out_whole"]) < 1e-7 and np.float32(ph) == GOLD["shift_phase_whole"]
    y, st = oracle.decimating_shift_addition_cc(GOLD["shift_in"][:448], 0.01, 2, 1, 0.5)
    assert rel_rms(y, GOLD["dshift_out"]) < 1e-7
    assert st[0] == int(GOLD["dshift_state"][0]) and np.float32(st[1]) == np.float32(GOLD["dshift_state"][1])


def test_golden_fir(oracle):
    for key, d, taps in (("fir_out_79_d10", 10, "lowpass_79"), ("fir_out_199_d10", 10, "lowpass_199")):
        y = oracle.fir_decimate_cc(GOLD["fir_in"], d, GOLD[taps])
        assert y.size == GOLD[key].size and rel_rms(y, GOLD[key]) < TIGHT
    y = oracle.fir_decimate_cc(GOLD["fir_in"][:1000], 7, GOLD["lowpass_79"])
    assert y.size == GOLD["fir_out_79_d7"].size == (1000 - 79) // 7 + 1
    assert rel_rms(y, GOLD["fir_out_79_d7"]) < TIGHT


def test_golden_fmdemod(oracle):
    y, last = oracle.fmdemod_quadri_cf(GOLD["fm_in"], 0.25 - 0.5j)
    assert np.array_equal(y, GOLD["fm_out"]) and np.complex64(last) == GOLD["fm_last"]


def test_golden_fractional_decimator(oracle):
    y = oracle.fractional_decimator_ff(GOLD["fd_in"], 5.0, 12, None, 1024)
    assert y.size == GOLD["fd_out_r5_blk1024"].size and rel_rms(y, GOLD["fd_out_r5_blk1024"]) < TIGHT
    y = oracle.fractional_decimator_ff(GOLD["fd_in"], 2.7183, 12, None, None)
    assert y.size == GOLD["fd_out_r2p7_whole"].size and rel_rms(y, GOLD["fd_out_r2p7_whole"]) < TIGHT
    y = oracle.fractional_decimator_ff(GOLD["fd_in"][:3000], 3.0, 4, oracle.firdes_lowpass_f(31, 0.15), None)
    assert y.size == GOLD["fd_out_r3_pts4_prefilter"].size and rel_rms(y, GOLD["fd_out_r3_pts4_prefilter"]) < TIGHT


def test_golden_fastagc(oracle):
    assert rel_rms(oracle.fastagc_ff(GOLD["agc_in"], 256, 1.0), GOLD["agc_out_b256"]) < 1e-7
    assert rel_rms(oracle.fastagc_ff(GOLD["agc_in"], 512, 0.5), GOLD["agc_out_b512_ref0p5"]) < 1e-7
    y = oracle.fastagc_ff(GOLD["agc_in"], 256, 1.0)
    assert not y[:512].any()                     # two blocks of latency: calloc'ed history (csdr.c:1394-1395)


def test_golden_audio_tail(oracle):
    y, last = oracle.deemphasis_wfm_ff(GOLD["deemph_in"], 50e-6, 48000, 0.0, 1024)
    assert np.array_equal(y, GOLD["deemph_out_50us_48k"]) and np.float32(last) == GOLD["deemph_last"]
    assert np.array_equal(oracle.limit_ff(GOLD["deemph_in"], 1.0), GOLD["limit_out"])


def _sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _at(y, key):
    """(y at the positions where the reference's output is stored, the stored values); the lengths must match"""
    n, want = int(REF[key + "_n"]), REF[key]
    assert y.size == n, (key, y.size, n)
    return y[pick_idx(n, want.size)], want


def test_ref_audio_tail(oracle):
    x = np.random.default_rng(21).uniform(-2, 2, 1 << 16).astype(np.float32)
    x[7] = np.nan; x[9] = np.inf; x[11] = -np.inf
    assert _sha(oracle.limit_ff(x, 0.7)) == REF["limit_0p7_sha"]                    # NaN -> +max like the reference build (minss/maxss)
    x = np.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)
    for i, (tau, fs, last, blk) in enumerate(((50e-6, 48000, 0.0, 1024), (75e-6, 240000, float("nan"), None), (50e-6, 44100, 0.3, 4096))):
        ya, la = oracle.deemphasis_wfm_ff(x, tau, fs, last, blk)
        assert _sha(ya) == REF[f"deemph_wfm_{i}_sha"] and np.float32(la) == REF[f"deemph_wfm_{i}_last"]


def test_ref_nco_deltas_over_many_rates(oracle):
    """shift_addition_init / decimating_shift_addition_init: the shipped build evaluates the deltas with sincosf (a -ffast-math narrowing); the
    oracle makes the same call and must agree bit for bit for every rate, because the recursion amplifies a one-ulp delta to ~3e-5."""
    rng = np.random.default_rng(0)
    rates = np.concatenate([rng.uniform(-0.5, 0.5, 6000), rng.uniform(-5, 5, 500), [0, 0.25, -0.25, 0.5, -0.5, 1e-7, -1e-7]]).astype(np.float32)
    assert _sha(np.array([oracle.shift_addition_init(float(rate)) for rate in rates], np.float32)) == REF["nco_deltas_sha"]


def test_golden_and_ref_deemphasis_nfm(oracle):
    """8(f) rank 1: the oracle's FIR on the tables the compiled reference exports (golden copies) reproduces the reference's outputs,
    on the stored vectors and on the reference's outputs for a longer seeded input; when oracle/_ref is built, the tables read out of it too."""
    for rate in (48000, 44100, 11025, 8000):
        taps = GOLD[f"nfm_taps_{rate}"]
        assert taps.size == {48000: 201, 44100: 123, 11025: 81, 8000: 81}[rate]
        y = oracle.deemphasis_nfm_ff(GOLD["nfm_in"], taps)
        assert y.size == GOLD["nfm_in"].size - taps.size and rel_rms(y, GOLD[f"nfm_out_{rate}"]) < 1e-6
    assert oracle.deemphasis_nfm_ff(GOLD["nfm_in"][:201], GOLD["nfm_taps_48000"]).size == 0
    x = np.random.default_rng(4).uniform(-1, 1, 20_000).astype(np.float32)
    for rate in (48000, 44100, 11025, 8000):
        assert rel_rms(*_at(oracle.deemphasis_nfm_ff(x, GOLD[f"nfm_taps_{rate}"]), f"nfm_{rate}")) < 1e-6
    assert REF["nfm_22050_n"] == 0                                                  # no table for that rate: the reference writes nothing
    if have_ref():
        from oracle.pyoracle import Ref
        r = Ref()
        for rate in r.NFM_RATES:
            assert np.array_equal(r.deemphasis_nfm_taps(rate), GOLD[f"nfm_taps_{rate}"])


def test_golden_and_ref_shift_addfast(oracle):
    """8(f) rank 3: given the reference's step table the oracle's recursion is bit-exact; the strict init is within 1 ulp of the
    reference build's (whose -ffast-math init goes through libmvec), which the 256-step recursion turns into < 1e-5 per 1024-call."""
    import ctypes as C
    from oracle.pyoracle import _CF, _p
    x = GOLD["shift_in"]; y = np.zeros_like(x); ph = 0.0
    steps = np.ascontiguousarray(GOLD["addfast_steps"])
    for s0 in range(0, x.size, 1024):
        ph = oracle.L.oracle_shift_addfast_cc(_p(x[s0:], _CF), _p(y[s0:], _CF), min(1024, x.size - s0), _p(steps, C.c_float), ph)
    assert np.array_equal(y, GOLD["addfast_out"]) and np.float32(ph) == GOLD["addfast_phase"]
    mine = oracle.shift_addfast_init(-0.085)
    assert np.abs(mine.view(np.int32) - steps.view(np.int32)).max() <= 1 and mine[8] == steps[8]
    y2, ph2 = oracle.shift_addfast_cc(x, -0.085, 0.0, 1024)
    assert rel_rms(y2, GOLD["addfast_out"]) < 1e-5 and np.float32(ph2) == GOLD["addfast_phase"]
    z = (np.random.default_rng(8).standard_normal(20_000) + 1j * np.random.default_rng(9).standard_normal(20_000)).astype(np.complex64)
    for rate in (0.25, 0.125):                                            # rates where both inits agree: only a call's seed can differ by
        assert np.array_equal(oracle.shift_addfast_init(rate), REF[f"addfast_init_{rate}"])    # an ulp (the -ffast-math build seeds with sincosf)
        for chunk in (1024, 4096, None):
            a, pa = oracle.shift_addfast_cc(z, rate, 0.3, chunk)
            assert rel_rms(*_at(a, f"addfast_{rate}_{chunk}")) < 1e-7 and np.float32(pa) == REF[f"addfast_{rate}_{chunk}_phase"], (rate, chunk)
    a, pa = oracle.shift_addfast_cc(z, 0.25, -1.0, 1022)                  # n % 4 tails stay untouched
    assert rel_rms(*_at(a, "addfast_1022")) < 1e-6 and np.float32(pa) == REF["addfast_1022_phase"]
    assert np.all(a[1020:1022] == 0) and np.all(REF["addfast_1022_tail"] == 0)


def test_ref_shift_table_bit_exact(oracle):
    """8(f) rank 3: with the reference's own table, the oracle's restatement of the BUILD's index arithmetic gives identical samples and phases
    (the reference's tables are stored as their ulp steps from the oracle's, its outputs on all cases as one digest per table size)"""
    x = (np.random.default_rng(1).standard_normal(60_000) + 1j * np.random.default_rng(2).standard_normal(60_000)).astype(np.complex64)
    for size in (65536, 1024, 100):
        mine = oracle.shift_table_init(size)
        t = (mine.view(np.int32) + REF[f"table_{size}_ulps"]).astype(np.int32).view(np.float32)
        assert np.abs(t - mine).max() <= 1.2e-7                                    # the build's sin() is libmvec's: an ulp here and there
        outs = []
        for rate in (-0.5, -0.31, -0.085, 0.0, 1e-4, 0.2, 0.25, 0.4999, 0.5):
            for ph0 in (0.0, 3.0, 1.5707964, 6.2831855):
                a, pa, _bad = oracle.shift_table_cc(x, rate, t, ph0)
                outs += [a.tobytes(), np.float32(pa).tobytes()]
        assert hashlib.sha256(b"".join(outs)).hexdigest() == REF[f"table_{size}_sha"], size


def test_golden_and_ref_shift_math(oracle):
    y, ph = oracle.shift_math_cc(GOLD["shift_in"], -0.085, -7.5, 1024)
    assert np.float32(ph) == GOLD["math_phase"] and rel_rms(y, GOLD["math_out"]) < TIGHT     # phase chain bit-exact; seeds: sincosf in the build
    z = (np.random.default_rng(8).standard_normal(30_000) + 1j * np.random.default_rng(9).standard_normal(30_000)).astype(np.complex64)
    for i, rate in enumerate((-0.5, -0.31, 0.0, 1e-4, 0.2, 0.4999, 0.5)):
        for j, (ph0, chunk) in enumerate(((0.0, 1024), (3.0, None), (-7.5, 1000), (100.0, 1024))):
            a, pa = oracle.shift_math_cc(z, rate, ph0, chunk)
            assert np.float32(pa) == REF[f"math_{i}_{j}_phase"] and rel_rms(*_at(a, f"math_{i}_{j}")) < TIGHT, (rate, ph0, chunk)


def test_ref_ima_adpcm(oracle):
    """8(f) rank 4: the oracle's IMA ADPCM encoder against the compiled reference's (bytes and carried state), and the waterfall line
    compression against the reference CLI's output"""
    rng = np.random.default_rng(0)
    for n in (2, 10, 1000, 4097):
        x = (rng.standard_normal(n) * rng.choice([10, 300, 5000, 40000])).clip(-32768, 32767).astype(np.int16)
        a, sa = oracle.encode_ima_adpcm_i16_u8(x, 3, -200)
        assert _sha(a) == REF[f"ima_{n}_sha"] and sa == tuple(REF[f"ima_{n}_state"])
    fft_size, frames = 512, 5
    db = rng.uniform(-120, -20, (frames, fft_size)).astype(np.float32)
    got = REF["adpcm_lines_512"]; want = oracle.compress_fft_adpcm_f_u8(db, fft_size).reshape(-1)
    assert np.array_equal(got[:want.size], want) and got.size == want.size


def test_golden_spectrum_and_unroll(oracle, ref=None):
    assert rel_rms(oracle.precalculate_window(1024, "HAMMING"), GOLD["win_hamming_1024"]) < TIGHT
    assert np.abs(oracle.logpower_cf(GOLD["spec_in"], -70.0) - GOLD["logpower_out"]).max() < 2e-5          # dB; an ulp at |x| ~ 100
    assert np.abs(oracle.logaveragepower_cf(GOLD["spec_in"], -70.0, 512, 4) - GOLD["logavg_out"]).max() < 2e-5
    y, ph = oracle.shift_unroll_cc(GOLD["shift_in"], -0.085, 0.0, 1024)
    assert rel_rms(y, GOLD["unroll_out"]) < 1e-7 and np.float32(ph) == GOLD["unroll_phase"]


def test_golden_bandpass_fir_fft(oracle):
    y = oracle.bandpass_fir_fft_cc(GOLD["bp_in"], -0.1, 0.2, 0.05)
    assert y.size == GOLD["bp_out"].size == (GOLD["bp_in"].size // 178) * 178     # 79 taps -> fft 256, 178 per block
    assert rel_rms(y, GOLD["bp_out"]) < 2e-6


def test_golden_fastddc(oracle):
    keys = [str(k) for k in GOLD["ddc_keys"]]
    for case, row in zip(GOLD["ddc_cases"], GOLD["ddc_geometry"]):
        geo = oracle.fastddc_geometry(float(case[0]), int(case[1]), float(case[2]))
        for k, v in zip(keys, row):
            assert np.float32(geo[k]) == np.float32(v), (case, k, geo[k], v)
    geo = oracle.fastddc_geometry(0.002, 64, 0.1)   # BASELINE config 3 geometry quoted in SURVEY 8(a) a11
    assert (geo["fft_size"], geo["taps_length"], geo["input_size"], geo["pre_decimation"], geo["post_decimation"],
            geo["fft_inv_size"], geo["scrap"], geo["post_input_size"], geo["v"]) == (16384, 2049, 14336, 32, 2, 512, 64, 448, 8)
    ddc, err = oracle.fastddc_init(0.05, 8, 0.123)
    assert not err
    spectra = oracle.fastddc_fwd(GOLD["ddc_in"], ddc)
    assert rel_rms(np.stack(spectra), GOLD["ddc_fwd_out"]) < TIGHT
    y = oracle.fastddc_inv(list(GOLD["ddc_fwd_out"]), 0.05, 8, 0.123)
    assert y.size == GOLD["ddc_inv_out"].size and rel_rms(y, GOLD["ddc_inv_out"]) < 2e-6


# ------------------------------------------------------------------ the compiled reference, larger inputs
def _cplx(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


def test_ref_conversions_all_codes(oracle):
    u8 = np.arange(256, dtype=np.uint8)
    s16 = np.arange(-32768, 32768).astype(np.int16)
    f = np.random.default_rng(3).uniform(-1, 1, 1 << 18).astype(np.float32)
    assert _sha(oracle.convert_u8_f(u8)) == REF["conv_u8_sha"]
    assert _sha(oracle.convert_s16_f(s16)) == REF["conv_s16_sha"]
    assert _sha(oracle.convert_f_s16(f)) == REF["conv_f_s16_sha"]


@pytest.mark.parametrize("T,D,bw", [(79, 10, 0.05), (199, 10, 0.0201), (801, 50, 0.005)])
def test_ref_fir_decimate(oracle, T, D, bw):
    assert oracle.firdes_filter_len(bw) == REF[f"firdes_len_{T}"] == T
    taps = REF[f"firdes_taps_{T}"]
    assert rel_rms(oracle.firdes_lowpass_f(T, 0.5 / D), taps) < TIGHT
    x = _cplx(np.random.default_rng(T), 262144)
    ya = oracle.fir_decimate_cc(x, D, taps)
    assert ya.size == (x.size - T) // D + 1
    assert rel_rms(*_at(ya, f"fir_dec_{T}")) < TIGHT


SHIFT_CASES = [(-0.085, 1024), (0.2, 1024), (0.4999, 1024), (0.01, 16384), (-0.3, None)]


@pytest.mark.parametrize("rate,chunk", SHIFT_CASES)
def test_ref_shift_addition(oracle, rate, chunk):
    i = SHIFT_CASES.index((rate, chunk))
    x = _cplx(np.random.default_rng(7), 1 << 17)
    ya, pa = oracle.shift_addition_cc(x, rate, 0.0, chunk)
    assert np.float32(pa) == REF[f"shift_add_{i}_phase"]
    assert rel_rms(*_at(ya, f"shift_add_{i}")) < 1e-7            # identical recursion; only the seed cos/sin may differ by an ulp


def test_ref_fmdemod_fracdec_agc(oracle):
    rng = np.random.default_rng(11)
    t = np.arange(1 << 16)
    fm = np.exp(1j * np.cumsum(0.4 * np.sin(2 * np.pi * t / 300))).astype(np.complex64)
    ya, la = oracle.fmdemod_quadri_cf(fm)
    assert _sha(ya) == REF["fmdemod_sha"] and np.complex64(la) == REF["fmdemod_last"]
    aud = rng.uniform(-1, 1, 1 << 16).astype(np.float32)
    for i, (rate, blk) in enumerate(((5.0, 1024), (5.0, None), (1.5, 1024), (48.0 / 44.1, 4096))):
        ya = oracle.fractional_decimator_ff(aud, rate, 12, None, blk)
        assert rel_rms(*_at(ya, f"fracdec_{i}")) < TIGHT, (rate, blk)
    for i, (block, refl) in enumerate(((1024, 1.0), (100, 0.3))):
        ya = oracle.fastagc_ff(aud * 0.05, block, refl)
        assert rel_rms(*_at(ya, f"agc_{i}")) < 1e-7


def test_ref_fft_paths(oracle):
    rng = np.random.default_rng(13)
    x = _cplx(rng, 2098 * 4)
    ya = oracle.bandpass_fir_fft_cc(x, -0.05, 0.05, 0.002)
    assert ya.size == 2098 * 4 and rel_rms(*_at(ya, "fft_bandpass")) < 2e-6
    ddc, _ = oracle.fastddc_init(0.002, 64, -0.2)
    xs = _cplx(rng, ddc.input_size * 2)
    sa = oracle.fastddc_fwd(xs, ddc)
    assert rel_rms(*_at(np.stack(sa).reshape(-1), "fft_ddc_fwd")) < TIGHT
    ya = oracle.fastddc_inv(sa, 0.002, 64, -0.2); yb = REF["fft_ddc_inv"]
    assert ya.size == yb.size == 2 * 224 and rel_rms(ya, yb) < 2e-6
