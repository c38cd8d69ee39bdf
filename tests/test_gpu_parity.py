"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI of
libcsdr_b200.so, against the CPU oracle (oracle/liboracle.so), the committed golden vectors and -- when
present as a prebuilt binary -- the compiled reference itself (oracle/_ref/libcsdr_ref.so).

Tolerances (BASELINE.json north_star): bit-exact for convert_u8_f / convert_f_s16 (and convert_s16_f);
<= 1e-5 relative RMS per channel for float blocks.  Tight internal bars (1e-6) are used where the GPU
performs the same rounding sequence as the oracle.
"""
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_golden.npz")
REF = np.load(Path(__file__).parent / "golden" / "ref_outputs.npz")         # the compiled reference on the seeded inputs below (make_ref_outputs.py)
NORTH_STAR_TOL = 1e-5


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device; refusing to fall back to anything else")
    import csdr_b200
    csdr_b200.lib()          # raises if the .so is missing: the product path must fail loudly
    return csdr_b200


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cplx(rng, n, amp=1.0):
    return ((rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)) * amp).astype(np.complex64)


def _rel(y, ref):
    from oracle.pyoracle import rel_rms
    return rel_rms(y, ref)


def _at(y, key):
    """(y at the positions where the reference's output is stored, the stored values); the lengths must match"""
    from oracle.pyoracle import pick_idx
    n, want = int(REF[key + "_n"]), REF[key]
    assert y.size == n, (key, y.size, n)
    return y[pick_idx(n, want.size)], want


# ------------------------------------------------------------------------------------------ K1
def test_convert_u8_f_bit_exact(gpu, oracle):
    x = np.concatenate([np.arange(256, dtype=np.uint8), np.random.default_rng(0).integers(0, 256, 2_000_003).astype(np.uint8)])
    y = gpu.convert_u8_f(_dev(x)).cpu().numpy()
    assert np.array_equal(y, oracle.convert_u8_f(x))
    assert np.array_equal(y[:256], GOLD["u8_out"])
    # host-pointer drop-in, odd sizes
    for n in (1, 15, 16, 17, 1024, 4099):
        assert np.array_equal(gpu.libcsdr.convert_u8_f(x[:n]), oracle.convert_u8_f(x[:n]))


def test_convert_s16_both_ways_bit_exact(gpu, oracle):
    s = np.arange(-32768, 32768).astype(np.int16)
    assert np.array_equal(gpu.convert_s16_f(_dev(s)).cpu().numpy(), oracle.convert_s16_f(s))
    assert np.array_equal(gpu.libcsdr.convert_s16_f(GOLD["s16_in"]), GOLD["s16_out"])
    f = np.concatenate([GOLD["f_in"], np.random.default_rng(1).uniform(-1, 1, 1_000_001).astype(np.float32),
                        np.array([3e9, -3e9, np.nan, np.inf, -np.inf, 1.00001, -1.00001], np.float32)])
    assert np.array_equal(gpu.convert_f_s16(_dev(f)).cpu().numpy(), oracle.convert_f_s16(f))
    assert np.array_equal(gpu.libcsdr.convert_f_s16(GOLD["f_in"]), GOLD["f_s16_out"])


# ------------------------------------------------------------------------------------------ K3
@pytest.mark.parametrize("variant", [-1, 0, 1, 2, 3, 4, 5, 6, 7])
def test_fir_bank_headline_shape_vs_oracle(gpu, oracle, variant):
    """256-channel geometry of BASELINE config 2 (T=199, D=10) at an oracle-sized N, every tiling variant."""
    T, D, C, N = 199, 10, 8, 40_000 + 7
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    assert _rel(taps, oracle.firdes_lowpass_f(T, 0.5 / D)) < 1e-6
    x = np.stack([_cplx(np.random.default_rng(c), N) for c in range(C)])
    y = gpu.fir_decimate_bank_cc(_dev(x), D, taps, variant=variant).cpu().numpy()
    assert y.shape == (C, (N - T) // D + 1)
    for c in range(C):
        assert _rel(y[c], oracle.fir_decimate_cc(x[c], D, taps)) < 1e-6, c


@pytest.mark.parametrize("T,D,N", [(79, 10, 16384), (199, 10, 16384), (199, 10, 199), (199, 10, 198), (199, 10, 208), (199, 10, 209),
                                   (79, 7, 5000), (801, 50, 70000), (33, 3, 1001), (5, 1, 64), (200, 10, 30011), (123, 10, 9999)])
def test_fir_bank_edge_geometries(gpu, oracle, T, D, N):
    taps = np.random.default_rng(T).uniform(-1, 1, T).astype(np.float32) / T
    x = np.stack([_cplx(np.random.default_rng(100 + c), N) for c in range(3)])
    n_out = (N - T) // D + 1 if N >= T else 0
    if n_out == 0:
        assert gpu.fir_out_len(N, D, T) == 0
        assert gpu.libcsdr.fir_decimate_cc(x[0], D, taps).size == 0
        return
    y = gpu.fir_decimate_bank_cc(_dev(x), D, taps).cpu().numpy()
    assert y.shape == (3, n_out)
    for c in range(3):
        assert _rel(y[c], oracle.fir_decimate_cc(x[c], D, taps)) < 2e-6
    # host-pointer drop-in on one channel
    assert _rel(gpu.libcsdr.fir_decimate_cc(x[1], D, taps), oracle.fir_decimate_cc(x[1], D, taps)) < 2e-6


def test_fir_golden_and_reference(gpu):
    for key, taps in (("fir_out_79_d10", "lowpass_79"), ("fir_out_199_d10", "lowpass_199")):
        y = gpu.libcsdr.fir_decimate_cc(GOLD["fir_in"], 10, GOLD[taps])
        assert y.size == GOLD[key].size and _rel(y, GOLD[key]) < NORTH_STAR_TOL / 5
    x = _cplx(np.random.default_rng(5), 262144)
    taps = REF["fir_taps_199_0p05"]
    y = gpu.fir_decimate_bank_cc(_dev(x[None, :]), 10, taps).cpu().numpy()[0]
    assert _rel(*_at(y, "fir_262144_d10")) < NORTH_STAR_TOL / 5


def test_fir_bank_full_size_properties(gpu):
    """BASELINE config 2 at full size (256 x 2.4 M cf32): size-independent checks.
    (1) linearity: FIR(a*x1 + x2) == a*FIR(x1) + FIR(x2) to float rounding;
    (2) a DC input gives sum(taps) == 1; (3) spot outputs against a float64 dot product."""
    C, N, T, D = 256, 2_400_000, 199, 10
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.rand((C, N, 2), generator=g, device="cuda", dtype=torch.float32) * 2 - 1
    y = gpu.fir_decimate_bank_cc(x, D, taps)
    n_out = (N - T) // D + 1
    assert y.shape == (C, n_out)
    idx = np.random.default_rng(9).integers(0, n_out, 64)
    t64 = torch.from_numpy(taps.astype(np.float64)).cuda()
    for c in (0, 1, 127, 255):
        for o in idx[:16]:
            seg = x[c, o * D:o * D + T].double()
            want = (seg * t64[:, None]).sum(0)
            got = torch.view_as_real(y[c, o]).double()
            assert torch.allclose(got, want, atol=2e-6, rtol=0), (c, o)
    assert torch.view_as_real(y[:, -1]).abs().max() < 1.0       # last valid output written, finite and sane
    del y
    x2 = x[:8, :200_000].contiguous()
    ya = gpu.fir_decimate_bank_cc(x2, D, taps)
    yb = gpu.fir_decimate_bank_cc((x2 * 0.5 + 0.25).contiguous(), D, taps)
    lin = ya * 0.5 + torch.complex(torch.tensor(0.25, device="cuda"), torch.tensor(0.25, device="cuda"))
    assert (yb - lin).abs().max() < 5e-6


# ------------------------------------------------------------------------------------------ K4
def test_fmdemod_quadri(gpu, oracle):
    t = np.arange(100_003)
    fm = np.exp(1j * np.cumsum(0.4 * np.sin(2 * np.pi * t / 300))).astype(np.complex64)
    x = np.stack([fm, np.roll(fm, 17) * 0.5, _cplx(np.random.default_rng(2), fm.size)])
    x[2, 100:110] = 0                                                 # den == 0 -> exact zeros
    last = np.array([0.25 - 0.5j, 0, 1 + 1j], np.complex64)
    y, lo = gpu.fmdemod_quadri_bank_cf(_dev(x), last=_dev(last), return_last=True)
    y = y.cpu().numpy(); lo = lo.cpu().numpy()
    for c in range(3):
        want, wl = oracle.fmdemod_quadri_cf(x[c], complex(last[c]))
        assert _rel(y[c], want) < 1e-6 and np.complex64(wl) == lo[c]
        assert np.abs(y[c] - want).max() <= 2e-7 * max(1.0, np.abs(want).max())
    assert not y[2, 101:110].any()
    yg, lg = gpu.libcsdr.fmdemod_quadri_cf(GOLD["fm_in"], 0.25 - 0.5j)
    assert _rel(yg, GOLD["fm_out"]) < 1e-6 and np.complex64(lg) == GOLD["fm_last"]
