"""GPU parity tests, part 2 (-m gpu): K2 shift, K5 fractional decimator, K6 fastagc, K7 FFT, K9 overlap-add bank,
K8 fastddc -- bank API and libcsdr drop-ins, all through the C ABI, against the oracle / compiled reference / golden vectors.
Float tolerance of the north star: 1e-5 relative RMS; tighter internal bars where the GPU replays the same roundings."""
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_golden.npz")
REF = np.load(Path(__file__).parent / "golden" / "ref_outputs.npz")         # the compiled reference on the seeded inputs below (make_ref_outputs.py)
TOL = 1e-5


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import csdr_b200
    csdr_b200.lib()
    return csdr_b200


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cplx(rng, n, amp=1.0):
    return ((rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)) * amp).astype(np.complex64)


def _at(y, key):
    """(y at the positions where the reference's output is stored, the stored values); the lengths must match"""
    from oracle.pyoracle import pick_idx
    n, want = int(REF[key + "_n"]), REF[key]
    assert y.size == n, (key, y.size, n)
    return y[pick_idx(n, want.size)], want


def _rel(y, ref):
    from oracle.pyoracle import rel_rms
    return rel_rms(y, ref)


# ------------------------------------------------------------------------------------------ K2
@pytest.mark.parametrize("chunk,N", [(1024, 16384), (1024, 16384 + 777), (1000, 50_000), (4096, 4096), (0, 3000), (37, 1000)])
def test_shift_bank_replays_reference_state_chain(gpu, oracle, chunk, N):
    rng = np.random.default_rng(N)
    rates = np.array([-0.085, 0.2, 0.4999, 0.0123, -0.3, 1e-4, 0.25], np.float32)
    x = _cplx(rng, N)
    y, ph = gpu.shift_addition_bank_cc(_dev(x), rates, chunk=chunk)                 # one shared wideband input
    y = y.cpu().numpy(); ph = ph.cpu().numpy()
    for c, r in enumerate(rates):
        want, wp = oracle.shift_addition_cc(x, float(r), 0.0, chunk if chunk > 0 else None)
        assert np.float32(wp) == ph[c], (c, wp, ph[c])
        assert _rel(y[c], want) < 1e-7, c                                           # same recursion; seeds may differ by an ulp
    # continue the stream: phases carried over, per-channel inputs this time
    x2 = np.stack([_cplx(np.random.default_rng(c), 5000) for c in range(rates.size)])
    y2, ph2 = gpu.shift_addition_bank_cc(_dev(x2), rates, phases=_dev(ph), chunk=1024)
    for c, r in enumerate(rates):
        want, wp = oracle.shift_addition_cc(x2[c], float(r), float(ph[c]), 1024)
        assert _rel(y2[c].cpu().numpy(), want) < 1e-7 and np.float32(wp) == ph2[c].item()


def test_shift_dropin_and_golden(gpu, oracle):
    y, ph = gpu.libcsdr.shift_addition_cc(GOLD["shift_in"], -0.085, 0.0, 1024)
    assert _rel(y, GOLD["shift_out_chunk1024"]) < 1e-7 and np.float32(ph) == GOLD["shift_phase_chunk1024"]
    y, ph = gpu.libcsdr.shift_addition_cc(GOLD["shift_in"], 0.2, 0.3, None)
    assert _rel(y, GOLD["shift_out_whole"]) < 1e-7 and np.float32(ph) == GOLD["shift_phase_whole"]
    x = _cplx(np.random.default_rng(3), 1 << 16)
    ya, pa = gpu.libcsdr.shift_addition_cc(x, -0.3, 0.0, None)                       # one 65536-step chain like test200.c:101
    assert _rel(*_at(ya, "shift_65536_m0p3")) < 1e-7 and np.float32(pa) == REF["shift_65536_m0p3_phase"]
    yd, st = gpu.libcsdr.decimating_shift_addition_cc(GOLD["shift_in"][:448], 0.01, 2, 1, 0.5)
    assert _rel(yd, GOLD["dshift_out"]) < 1e-7
    assert st[0] == int(GOLD["dshift_state"][0]) and np.float32(st[1]) == np.float32(GOLD["dshift_state"][1])
    for n, d, rem in ((1000, 7, 3), (448, 2, 0), (5, 10, 2), (100, 3, 99)):
        ya, sa = gpu.libcsdr.decimating_shift_addition_cc(x[:n], -0.07, d, rem, 1.0)
        yb, sb = oracle.decimating_shift_addition_cc(x[:n], -0.07, d, rem, 1.0)
        assert ya.size == yb.size and sa[0] == sb[0] and np.float32(sa[1]) == np.float32(sb[1])
        assert ya.size == 0 or _rel(ya, yb) < 1e-7


# ------------------------------------------------------------------------------------------ K5
@pytest.mark.parametrize("rate,pts,block", [(5.0, 12, 1024), (5.0, 12, None), (2.7183, 12, None), (1.5, 4, 512), (48.0 / 44.1, 12, 4096), (10.0, 2, None)])
def test_fractional_decimator_positions_are_exact(gpu, oracle, rate, pts, block):
    x = np.random.default_rng(int(rate * 100)).uniform(-1, 1, 40_000).astype(np.float32)
    want = oracle.fractional_decimator_ff(x, rate, pts, None, block)
    got = gpu.libcsdr.fractional_decimator_ff(x, rate, pts, None, block)
    assert got.size == want.size                                                    # one flipped ceilf() would change the count or shift everything
    assert np.array_equal(got, want)                                                # same IEEE operation order -> bit exact vs the strict oracle


def test_fractional_decimator_bank_prefilter_and_golden(gpu, oracle):
    got = gpu.libcsdr.fractional_decimator_ff(GOLD["fd_in"], 5.0, 12, None, 1024)
    assert got.size == GOLD["fd_out_r5_blk1024"].size and _rel(got, GOLD["fd_out_r5_blk1024"]) < 1e-6
    taps = oracle.firdes_lowpass_f(31, 0.15)
    got = gpu.libcsdr.fractional_decimator_ff(GOLD["fd_in"][:3000], 3.0, 4, taps, None)
    assert got.size == GOLD["fd_out_r3_pts4_prefilter"].size and _rel(got, GOLD["fd_out_r3_pts4_prefilter"]) < 1e-6
    x = np.stack([np.random.default_rng(c).uniform(-1, 1, 30_000).astype(np.float32) for c in range(5)])
    y, state = gpu.fractional_decimator_bank_ff(_dev(x), 5.0, 12)
    y = y.cpu().numpy(); state = state.cpu().numpy()
    for c in range(5):
        want = oracle.fractional_decimator_ff(x[c], 5.0, 12, None, None)
        assert state[c, 2] == want.size and np.array_equal(y[c, :want.size], want)


# ------------------------------------------------------------------------------------------ K6
def test_fastagc(gpu, oracle):
    assert _rel(gpu.libcsdr.fastagc_ff(GOLD["agc_in"], 256, 1.0), GOLD["agc_out_b256"]) < 1e-7
    assert _rel(gpu.libcsdr.fastagc_ff(GOLD["agc_in"], 512, 0.5), GOLD["agc_out_b512_ref0p5"]) < 1e-7
    rng = np.random.default_rng(4)
    env = np.repeat(rng.uniform(0.001, 1.0, 40).astype(np.float32), 1024)
    x = np.stack([rng.uniform(-1, 1, env.size).astype(np.float32) * env * s for s in (1.0, 0.01, 0.0, 30.0)])
    y, state, hist = gpu.fastagc_bank_ff(_dev(x), 1024, 1.0)
    y = y.cpu().numpy()
    for c in range(4):
        want = oracle.fastagc_ff(x[c], 1024, 1.0)
        assert np.array_equal(y[c], want), c                                         # same roundings (double ramp) -> bit exact
    assert not y[:, :2048].any()                                                    # two blocks of latency
    # streaming: feeding the same stream in two calls gives the same output
    half = 20 * 1024
    ya, st, hi = gpu.fastagc_bank_ff(_dev(x[:, :half]), 1024, 1.0)
    yb, _, _ = gpu.fastagc_bank_ff(_dev(x[:, half:]), 1024, 1.0, state=st, hist=hi)
    assert np.array_equal(np.concatenate([ya.cpu().numpy(), yb.cpu().numpy()], 1), y)
    y1, st1, hi1 = gpu.fastagc_bank_ff(_dev(x[:, :1024]), 1024, 1.0)                 # one block at a time like the CLI
    y2, st2, hi2 = gpu.fastagc_bank_ff(_dev(x[:, 1024:2048]), 1024, 1.0, state=st1, hist=hi1)
    y3, _, _ = gpu.fastagc_bank_ff(_dev(x[:, 2048:3072]), 1024, 1.0, state=st2, hist=hi2)
    assert np.array_equal(y3.cpu().numpy(), y[:, 2048:3072])


# ------------------------------------------------------------------------------------------ K7
@pytest.mark.parametrize("n", [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384])
def test_fft_all_sizes_vs_float64_dft(gpu, n):
    rng = np.random.default_rng(n)
    x = _cplx(rng, 3 * n).reshape(3, n)
    for inv in (False, True):
        y = gpu.fft_c2c(_dev(x), inverse=inv).cpu().numpy()
        want = np.fft.ifft(x.astype(np.complex128), axis=1) * n if inv else np.fft.fft(x.astype(np.complex128), axis=1)
        assert _rel(y, want) < 1e-6, (n, inv)                                       # ~1e-7*log2(n) from the exact DFT
    a = gpu.libcsdr.dft(x[0], True)
    assert _rel(a, np.fft.fft(x[0].astype(np.complex128))) < 1e-6


# ------------------------------------------------------------------------------------------ K9
def test_bandpass_fir_fft_dropin_golden_and_reference(gpu, oracle):
    y = gpu.libcsdr.bandpass_fir_fft_cc(GOLD["bp_in"], -0.1, 0.2, 0.05)
    assert y.size == GOLD["bp_out"].size and _rel(y, GOLD["bp_out"]) < TOL / 2
    x = _cplx(np.random.default_rng(6), 2098 * 5)
    y = gpu.libcsdr.bandpass_fir_fft_cc(x, -0.05, 0.05, 0.002)                      # BASELINE config 5 geometry: 1999 taps, 4096-pt, 2098/block
    assert _rel(*_at(y, "bandpass_cfg5")) < TOL / 2
    T = oracle.firdes_filter_len(0.002); taps = oracle.firdes_bandpass_c(T, -0.05, 0.05)
    direct = np.convolve(x.astype(np.complex128), taps.astype(np.complex128))[:y.size]
    assert _rel(y, direct) < TOL / 2


@pytest.mark.parametrize("bw,lo,hi,nblocks", [(0.002, -0.05, 0.05, 70), (0.05, 0.1, 0.3, 33), (0.005, -0.2, -0.1, 40)])
def test_bandpass_fir_fft_bank(gpu, oracle, bw, lo, hi, nblocks):
    T, N, isz, ov = gpu.bandpass_geometry(bw)                                        # (0.005 -> 801 taps, 1024-pt: overlap 800 > input 224)
    C = 5
    x = np.stack([_cplx(np.random.default_rng(c), nblocks * isz) for c in range(C)])
    tf = gpu.bandpass_taps_fft(lo, hi, bw)
    y, tail = gpu.bandpass_fir_fft_bank_cc(_dev(x), tf, isz)
    y = y.cpu().numpy()
    for c in range(C):
        assert _rel(y[c], oracle.bandpass_fir_fft_cc(x[c], lo, hi, bw)) < TOL / 2, c
    # block-size independence: the same stream in two calls with the tail carried
    cut = (nblocks // 3) * isz
    ya, ta = gpu.bandpass_fir_fft_bank_cc(_dev(x[:, :cut]), tf, isz)
    yb, _ = gpu.bandpass_fir_fft_bank_cc(_dev(x[:, cut:]), tf, isz, tail=ta)
    assert _rel(np.concatenate([ya.cpu().numpy(), yb.cpu().numpy()], 1), y) < 1e-7


# ------------------------------------------------------------------------------------------ K8
def test_fastddc_golden(gpu):
    ddc = gpu.fastddc_init(0.05, 8, 0.123)
    sp, _ = gpu.fastddc_fwd_cc(_dev(GOLD["ddc_in"]), ddc)
    assert _rel(sp.cpu().numpy(), GOLD["ddc_fwd_out"]) < 1e-6
    y = gpu.libcsdr.fastddc_inv(list(GOLD["ddc_fwd_out"]), 0.05, 8, 0.123)
    assert y.size == GOLD["ddc_inv_out"].size and _rel(y, GOLD["ddc_inv_out"]) < TOL / 2
    out, counts, _ = gpu.fastddc_inv_bank_cc(sp, [0.123], 8, 0.05)
    n = int(counts[0].item())
    assert n == GOLD["ddc_inv_out"].size and _rel(out[0, :n].cpu().numpy(), GOLD["ddc_inv_out"]) < TOL / 2


def test_fastddc_config3_bank_vs_oracle_and_reference(gpu, oracle):
    """BASELINE config 3 geometry: 16384-pt FFT, decimation 64, bw 0.002; several channels from one wideband stream."""
    bw, dec = 0.002, 64
    ddc = gpu.fastddc_init(bw, dec, 0.0)
    assert (ddc.fft_size, ddc.fft_inv_size, ddc.input_size, ddc.post_input_size, ddc.scrap) == (16384, 512, 14336, 448, 64)
    nblocks = 4
    n = nblocks * ddc.input_size
    rng = np.random.default_rng(8)
    shifts = [-0.4, -0.2113, 0.0, 0.1, 0.3337]
    t = np.arange(n)
    x = sum(np.exp(2j * np.pi * (s + 0.001) * t) for s in shifts).astype(np.complex64) / len(shifts) + _cplx(rng, n, 0.05)
    sp, ov = gpu.fastddc_fwd_cc(_dev(x), ddc)
    o_ddc, _ = oracle.fastddc_init(bw, dec, 0.0)
    want_sp = np.stack(oracle.fastddc_fwd(x, o_ddc))
    assert _rel(sp.cpu().numpy(), want_sp) < 1e-6
    out, counts, st = gpu.fastddc_inv_bank_cc(sp, shifts, dec, bw)
    for c, s in enumerate(shifts):
        want = oracle.fastddc_inv(list(want_sp), bw, dec, s)
        k = int(counts[c].item())
        assert k == want.size == nblocks * 224
        assert _rel(out[c, :k].cpu().numpy(), want) < TOL / 2, (c, s)
    rwant = REF["fastddc_cfg3_shift0p1"]
    assert _rel(out[3, :rwant.size].cpu().numpy(), rwant) < TOL / 2
    # streaming: second call continues phase/remain and the forward overlap
    x2 = _cplx(rng, 2 * ddc.input_size, 0.3)
    sp2, _ = gpu.fastddc_fwd_cc(_dev(x2), ddc, overlap=ov)
    out2, counts2, _ = gpu.fastddc_inv_bank_cc(sp2, shifts, dec, bw, state=st)
    xall = np.concatenate([x, x2])
    want_all = oracle.fastddc_inv(oracle.fastddc_fwd(xall, o_ddc), bw, dec, shifts[1])
    got = np.concatenate([out[1, :int(counts[1])].cpu().numpy(), out2[1, :int(counts2[1])].cpu().numpy()])
    assert got.size == want_all.size and _rel(got, want_all) < TOL / 2


def test_fastddc_odd_post_decimation(gpu, oracle):
    """decimation 6 -> pre 2, post 3: the remain counter of the post decimator walks between blocks."""
    bw, dec, s = 0.01, 6, 0.25
    ddc = gpu.fastddc_init(bw, dec, s)
    x = _cplx(np.random.default_rng(10), 5 * ddc.input_size)
    sp, _ = gpu.fastddc_fwd_cc(_dev(x), ddc)
    out, counts, _ = gpu.fastddc_inv_bank_cc(sp, [s, -0.1], dec, bw)
    o_ddc, _ = oracle.fastddc_init(bw, dec, s)
    for c, sh in enumerate([s, -0.1]):
        od, _ = oracle.fastddc_init(bw, dec, sh)
        want = oracle.fastddc_inv(oracle.fastddc_fwd(x, od), bw, dec, sh)
        k = int(counts[c])
        assert k == want.size and _rel(out[c, :k].cpu().numpy(), want) < TOL / 2


# ------------------------------------------------------------------------------------------ exact phase wrap + fused DDC bank
def test_phase_wrap_fast_forward_is_exact(gpu, oracle):
    """The binade-by-binade fast-forward of `while(ph>PI) ph-=2*PI` (common.cuh) must give the very float the loop gives.
    One shift_addition_cc call of n samples advances the phase by 2*rate*PI*n un-wrapped (up to ~2^20 here), then wraps it."""
    x = _cplx(np.random.default_rng(0), 64)
    for rate in (0.4999, -0.4999, 0.31, 0.123456, -0.25, 1e-3, 0.0401):
        for n in (64, 1000, 4099, 65536, 300_000):
            xx = np.resize(x, n)
            _, ph = gpu.shift_addition_bank_cc(_dev(xx), [rate], chunk=0)
            _, want = oracle.shift_addition_cc(xx, rate, 0.0, None)
            assert np.float32(want) == ph[0].item(), (rate, n, want, ph[0].item())
    # many consecutive wraps with carried phase: 3000 chunks of 64 samples
    xx = np.resize(x, 64 * 3000)
    for rate in (0.4999, -0.37):
        _, ph = gpu.shift_addition_bank_cc(_dev(xx), [rate], chunk=64)
        _, want = oracle.shift_addition_cc(xx, rate, 0.0, 64)
        assert np.float32(want) == ph[0].item()


@pytest.mark.parametrize("D,bw,demod", [(50, 0.005, True), (50, 0.005, False), (10, 0.0201, True), (10, 0.05, True)])
def test_fused_ddc_bank_matches_unfused_reference_chain(gpu, oracle, D, bw, demod):
    """BASELINE config 4 chain on a small bank: shift_addition_cc (1024-sample chunks) | fir_decimate_cc D | fmdemod_quadri_cf."""
    T = oracle.firdes_filter_len(bw)
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    N = 60_000 + 13
    rng = np.random.default_rng(D)
    t = np.arange(N)
    rates = np.array([-0.41, -0.27, -0.13, 0.01, 0.15, 0.29, 0.43], np.float32)     # one FM carrier per passband (den stays away from 0)
    wide = sum(0.3 * np.exp(1j * (2 * np.pi * (-float(r)) * t + np.cumsum(0.05 * np.sin(2 * np.pi * t / (2000.0 + 100 * k))))) for k, r in enumerate(rates))
    wide = (wide + 0.01 * (rng.normal(size=N) + 1j * rng.normal(size=N))).astype(np.complex64)
    out, ph, last = gpu.ddc_bank(_dev(wide), rates, D, taps, demod=demod, chunk=1024)
    out = out.cpu().numpy()
    n_out = (N - T) // D + 1
    assert out.shape == (rates.size, n_out)
    for c, r in enumerate(rates):
        sh, _ = oracle.shift_addition_cc(wide, float(r), 0.0, 1024)
        base = oracle.fir_decimate_cc(sh, D, taps)
        want = oracle.fmdemod_quadri_cf(base)[0] if demod else base
        # baseband: only the FIR summation order differs (~3e-7).  Discriminator output: its numerator is a cancellation, so the
        # same baseband noise is amplified; the bar is the north-star 1e-5 relative RMS on a properly modulated signal.
        assert _rel(out[c], want) < (TOL if demod else 2e-6), (c, r, _rel(out[c], want))
        if demod:
            assert _rel(np.array([last[c].item()]), base[-1:]) < 1e-5


def test_fused_ddc_bank_streams_block_by_block(gpu, oracle):
    """Two calls with the tail re-presented (csdr.c:1172-1174) and chunk phase/offset carried == one long reference stream."""
    D, T, chunk = 50, 801, 1024
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    rng = np.random.default_rng(3)
    N = 50_000
    t = np.arange(N)
    rates = np.array([0.123, -0.4], np.float32)
    wide = sum(0.4 * np.exp(1j * (2 * np.pi * (-float(r)) * t + np.cumsum(0.004 * np.sin(2 * np.pi * t / 5000.0)))) for r in rates)
    wide = (wide + 0.005 * (rng.normal(size=N) + 1j * rng.normal(size=N))).astype(np.complex64)     # one FM carrier per passband
    n1 = 20_000
    o1, ph1, last1 = gpu.ddc_bank(_dev(wide[:n1]), rates, D, taps, demod=True, chunk=chunk, offset=0)
    consumed = o1.shape[1] * D
    o2, ph2, last2 = gpu.ddc_bank(_dev(wide[consumed:]), rates, D, taps, demod=True, chunk=chunk, offset=consumed % chunk, phases=ph1, last=last1)
    got = np.concatenate([o1.cpu().numpy(), o2.cpu().numpy()], 1)
    for c, r in enumerate(rates):
        sh, _ = oracle.shift_addition_cc(wide, float(r), 0.0, chunk)
        want = oracle.fmdemod_quadri_cf(oracle.fir_decimate_cc(sh, D, taps))[0]
        assert got.shape[1] == want.size and _rel(got[c], want) < TOL


# ------------------------------------------------------------------------------------------ audio tail (8f rank 1)
def test_audio_tail_limit_and_deemphasis(gpu, oracle):
    x = np.random.default_rng(31).uniform(-2, 2, 200_003).astype(np.float32)
    x[7] = np.nan; x[9] = np.inf; x[11] = -np.inf
    assert np.array_equal(gpu.limit_ff(_dev(x), 0.7).cpu().numpy(), oracle.limit_ff(x, 0.7))
    assert np.array_equal(gpu.libcsdr.limit_ff(GOLD["deemph_in"], 1.0), GOLD["limit_out"])
    y, last = gpu.libcsdr.deemphasis_wfm_ff(GOLD["deemph_in"], 50e-6, 48000, 0.0, 1024)
    assert np.array_equal(y, GOLD["deemph_out_50us_48k"]) and np.float32(last) == GOLD["deemph_last"]     # same rounding sequence: bit exact
    xb = np.stack([np.random.default_rng(c).uniform(-1, 1, 50_001).astype(np.float32) for c in range(37)])
    lasts = np.linspace(-0.5, 0.5, 37).astype(np.float32); lasts[3] = np.nan
    yb, lb = gpu.deemphasis_wfm_bank_ff(_dev(xb), 75e-6, 240000, last=_dev(lasts))
    for c in range(37):
        want, wl = oracle.deemphasis_wfm_ff(xb[c], 75e-6, 240000, float(lasts[c]))
        assert np.array_equal(yb[c].cpu().numpy(), want) and np.float32(wl) == lb[c].item()


def test_ddc_bank_object_streams_with_lookahead(gpu, oracle):
    """csdrb_ddc_bank_*: many blocks with the tail re-presented, look-ahead pre-pass on the side stream, a block of a different size
    in the middle (look-ahead dropped) -- always equal to one long reference stream per channel."""
    D, T, chunk = 50, 801, 1024
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    rng = np.random.default_rng(17)
    N = 200_000
    t = np.arange(N)
    rates = np.array([0.123, -0.4, 0.31], np.float32)
    wide = sum(0.3 * np.exp(1j * (2 * np.pi * (-float(r)) * t + np.cumsum(0.004 * np.sin(2 * np.pi * t / 5000.0)))) for r in rates)
    wide = (wide + 0.005 * (rng.normal(size=N) + 1j * rng.normal(size=N))).astype(np.complex64)
    dwide = _dev(wide)
    bank = gpu.DdcBank(rates, D, taps, demod=True, chunk=chunk)
    pos, outs, sizes = 0, [], [30_000, 30_000, 30_000, 17_001, 30_000, 30_000]
    for sz in sizes:
        assert bank.offset == pos % chunk
        o = bank.process(dwide[pos:pos + sz])
        outs.append(o.cpu().numpy().copy())
        pos += o.shape[1] * D
    got = np.concatenate(outs, 1)
    for c, r in enumerate(rates):
        sh, _ = oracle.shift_addition_cc(wide[:pos + T], float(r), 0.0, chunk)
        want = oracle.fmdemod_quadri_cf(oracle.fir_decimate_cc(sh, D, taps))[0]
        assert _rel(got[c], want[:got.shape[1]]) < TOL, c
    bank.close()


# ------------------------------------------------------------------------------------------ spectrum path + shift_unroll (8f ranks 3, 4)
def test_spectrum_path_and_shift_unroll(gpu, oracle):
    assert np.array_equal(gpu.libcsdr.precalculate_window(1024, "HAMMING"), oracle.precalculate_window(1024, "HAMMING"))
    x = GOLD["spec_in"]
    assert np.abs(gpu.libcsdr.logpower_cf(x, -70.0) - GOLD["logpower_out"]).max() < 2e-5
    assert np.abs(gpu.libcsdr.logaveragepower_cf(x, -70.0, 512, 4) - GOLD["logavg_out"]).max() < 2e-5
    assert np.array_equal(gpu.libcsdr.apply_window_c(x[:1024], "BLACKMAN"), oracle.apply_precalculated_window_c(x[:1024], oracle.precalculate_window(1024, "BLACKMAN")))
    # whole-stream spectrum on the device vs window -> float64 DFT -> logpower on the CPU
    big = _cplx(np.random.default_rng(41), 64 * 2048, 0.5)
    db = gpu.spectrum_logpower(_dev(big), 2048, "HAMMING", -30.0).cpu().numpy()
    w = oracle.precalculate_window(2048, "HAMMING")
    for f in (0, 31, 63):
        want = oracle.logpower_cf(oracle.dft(oracle.apply_precalculated_window_c(big[f * 2048:(f + 1) * 2048], w)), -30.0)
        assert np.abs(db[f] - want).max() < 1e-3                                      # dB: FFT rounding (1e-7 relative) on bins far below the peak
    y, ph = gpu.libcsdr.shift_unroll_cc(GOLD["shift_in"], -0.085, 0.0, 1024)
    assert _rel(y, GOLD["unroll_out"]) < 1e-7 and np.float32(ph) == GOLD["unroll_phase"]
    xs = _cplx(np.random.default_rng(42), 20_000)
    rates = [0.2, -0.4999, 0.0123]
    yb, pb = gpu.shift_unroll_bank_cc(_dev(xs), rates)
    for c, r in enumerate(rates):
        want, wp = oracle.shift_unroll_cc(xs, r, 0.0, 1024)
        assert _rel(yb[c].cpu().numpy(), want) < 1e-7 and np.float32(wp) == pb[c].item()
