"""GPU tests (-m gpu) of the stdin/stdout command surface: our C host CLI (csdr_b200/csdr, computing on the GPU through
libcsdr_b200.so) against the UNMODIFIED reference CLI (oracle/_ref/csdr_ref, built from the reference's csdr.c) on the same
pipe graphs, plus the LD_PRELOAD drop-in: the reference's own binary running on top of our library.  Where the reference is not built, its
recorded outputs stand in for it (tests/reference_cli.py)."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from reference_cli import REFERENCE, arr, recorded, rel_rms

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = Path(__file__).resolve().parent.parent
OURS = ROOT / "csdr_b200" / "csdr"
LIB = ROOT / "csdr_b200" / "libcsdr_b200.so"
REF = ROOT / "oracle" / "_ref" / "csdr_ref"


@pytest.fixture(scope="module")
def clis():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    from csdr_b200.build import build
    build()
    assert OURS.exists() and LIB.exists()
    return str(OURS), str(REF) if REF.exists() else REFERENCE


@recorded
def run_graph(cli, stages, data: bytes, env=None, timeout=120) -> bytes:
    cmd = " | ".join(f"{cli} {s}" for s in stages)
    e = dict(os.environ); e.update(env or {})
    r = subprocess.run(["bash", "-c", cmd], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e, timeout=timeout)
    assert r.returncode == 0, (cmd, r.stderr[-2000:])
    return r.stdout


def rel(a, b):
    return rel_rms(a, b)


@recorded
def refuses(cli, stage, data: bytes) -> bool:
    """the command exits non-zero without writing anything"""
    r = subprocess.run(["bash", "-c", f"{cli} {stage}"], input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    return r.returncode != 0 and r.stdout == b""


def fm_u8(n, seed=0):
    """u8 IQ of an FM-modulated carrier + a little noise (so the discriminator has a defined output)."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    ph = np.cumsum(0.05 * np.sin(2 * np.pi * t / 4000.0)) + 2 * np.pi * 0.01 * t
    z = 0.7 * np.exp(1j * ph) + 0.01 * (rng.normal(size=n) + 1j * rng.normal(size=n))
    iq = np.empty(2 * n, np.float64); iq[0::2] = z.real; iq[1::2] = z.imag
    return np.clip(np.floor(iq * 127.5 + 128), 0, 255).astype(np.uint8).tobytes()


def test_config1_graph_matches_reference_cli(clis):
    """BASELINE configs[0]: convert_u8_f | fir_decimate_cc 10 0.05 HAMMING | fmdemod_quadri_cf on 1 M u8 IQ samples."""
    ours, ref = clis
    data = fm_u8(1_000_000)
    stages = ["convert_u8_f", "fir_decimate_cc 10 0.05 HAMMING", "fmdemod_quadri_cf"]
    a = arr(run_graph(ours, stages, data), np.float32)
    b = arr(run_graph(ref, stages, data), np.float32)
    assert a.size == b.size and a.size > 90_000                     # identical framing, including the stale tail blocks at EOF
    assert rel(a, b) < 1e-5
    # stage by stage: the byte conversion is bit-exact, framing identical
    a1 = run_graph(ours, stages[:1], data); b1 = run_graph(ref, stages[:1], data)
    assert a1 == b1
    a2 = arr(run_graph(ours, stages[:2], data), np.complex64); b2 = arr(run_graph(ref, stages[:2], data), np.complex64)
    assert a2.size == b2.size and rel(a2, b2) < 1e-5


def test_eof_framing_quirks(clis):
    ours, ref = clis
    for nbytes in (2048, 2000, 1, 1024, 5000):
        data = bytes(np.random.default_rng(nbytes).integers(0, 256, nbytes, dtype=np.uint8))
        a = run_graph(ours, ["convert_u8_f"], data); b = run_graph(ref, ["convert_u8_f"], data)
        assert len(a) == len(b), nbytes                              # e.g. 2048 B in -> 3 blocks (12288 B) out, 2000 B -> 2 blocks
        n = (nbytes // 1024) * 1024 * 4
        assert a[:n] == b[:n]
    x = np.random.default_rng(1).uniform(-1, 1, 40_000).astype(np.float32).tobytes()
    assert run_graph(ours, ["convert_f_s16"], x) == run_graph(ref, ["convert_f_s16"], x)
    s = np.random.default_rng(2).integers(-32768, 32767, 30_000).astype(np.int16).tobytes()
    assert run_graph(ours, ["convert_s16_f"], s) == run_graph(ref, ["convert_s16_f"], s)


def test_nfm_style_chain(clis):
    """shift | fir_decimate | fmdemod | fractional_decimator | fastagc | convert_f_s16 (the README.md:87 NFM graph minus limit/deemphasis)."""
    ours, ref = clis
    n = 600_000
    rng = np.random.default_rng(5)
    t = np.arange(n)
    z = (0.5 * np.exp(1j * (2 * np.pi * 0.2 * t + np.cumsum(0.02 * np.sin(2 * np.pi * t / 3000.0)))) +
         0.01 * (rng.normal(size=n) + 1j * rng.normal(size=n))).astype(np.complex64)
    stages = ["shift_addition_cc -0.2", "fir_decimate_cc 10 0.05 HAMMING", "fmdemod_quadri_cf", "fractional_decimator_ff 1.25", "fastagc_ff 1024 0.5"]
    a = arr(run_graph(ours, stages, z.tobytes()), np.float32)
    b = arr(run_graph(ref, stages, z.tobytes()), np.float32)
    assert a.size == b.size and a.size > 40_000
    assert rel(a, b) < 1e-5
    a16 = arr(run_graph(ours, stages + ["convert_f_s16"], z.tobytes()), np.int16)
    b16 = arr(run_graph(ref, stages + ["convert_f_s16"], z.tobytes()), np.int16)
    assert a16.size == b16.size and np.abs(a16.astype(np.int32) - b16.astype(np.int32)).max() <= 1     # float->short of values equal to 1e-5


def test_deemphasis_nfm_command(clis):
    """csdr.c:1068-1087: one block of look-behind before the first read, output in (block - taps) sized pieces, stale tail at EOF;
    unknown sample rate -> error exit like the reference."""
    ours, ref = clis
    for n in (50_000, 1024, 3000, 823):
        x = np.random.default_rng(n).uniform(-1, 1, n).astype(np.float32).tobytes()
        for rate in (48000, 11025):
            a = arr(run_graph(ours, [f"deemphasis_nfm_ff {rate}"], x), np.float32)
            b = arr(run_graph(ref, [f"deemphasis_nfm_ff {rate}"], x), np.float32)
            assert a.size == b.size and a.size > 0, (n, rate)
            assert rel(a, b) < 1e-5, (n, rate)
    for cli in (ours, ref):
        assert refuses(cli, "deemphasis_nfm_ff 22050", b"\0" * 8192)


def test_full_nfm_graph_of_the_readme(clis):
    """README.md:87 end to end: shift | fir_decimate 50 0.005 | fmdemod | limit | deemphasis_nfm 48000 | fastagc | convert_f_s16."""
    ours, ref = clis
    n = 2_400_000
    rng = np.random.default_rng(9)
    t = np.arange(n)
    audio = np.sin(2 * np.pi * 1000.0 / 2.4e6 * t) + 0.5 * np.sin(2 * np.pi * 2300.0 / 2.4e6 * t)
    z = (0.5 * np.exp(1j * (2 * np.pi * 0.145 * t + np.cumsum(2 * np.pi * 2500.0 / 2.4e6 * audio))) +
         0.002 * (rng.normal(size=n) + 1j * rng.normal(size=n))).astype(np.complex64)
    stages = ["shift_addition_cc -0.145", "fir_decimate_cc 50 0.005 HAMMING", "fmdemod_quadri_cf", "limit_ff", "deemphasis_nfm_ff 48000", "fastagc_ff"]
    a = arr(run_graph(ours, stages, z.tobytes()), np.float32)
    b = arr(run_graph(ref, stages, z.tobytes()), np.float32)
    assert a.size == b.size and a.size > 30_000
    assert rel(a, b) < 1e-5
    a16 = arr(run_graph(ours, stages + ["convert_f_s16"], z.tobytes()), np.int16)
    b16 = arr(run_graph(ref, stages + ["convert_f_s16"], z.tobytes()), np.int16)
    assert a16.size == b16.size and np.abs(a16.astype(np.int32) - b16.astype(np.int32)).max() <= 1


def test_shift_addfast_and_decimating_shift_commands(clis):
    """csdr.c:749-798 and 851-875.  shift_addfast: rates 0.25 / 0.125 are ones where the reference build's libmvec init equals the
    correctly rounded table, so the streams agree to seed level; at -0.085 the tables differ by one ulp, which 256 recursion steps
    per 1024-sample call turn into ~9e-6 -- still inside the 1e-5 bar (tests/test_oracle.py pins the same figure on the CPU)."""
    ours, ref = clis
    z = (np.random.default_rng(3).uniform(-1, 1, 100_000) + 1j * np.random.default_rng(4).uniform(-1, 1, 100_000)).astype(np.complex64).tobytes()
    for rate, bar in ((0.25, 1e-6), (0.125, 1e-6), (-0.085, 1e-5)):
        a = arr(run_graph(ours, [f"shift_addfast_cc {rate}"], z), np.complex64)
        b = arr(run_graph(ref, [f"shift_addfast_cc {rate}"], z), np.complex64)
        assert a.size == b.size and a.size > 0 and rel(a, b) < bar, (rate, rel(a, b))
    for rate, dec in ((0.1, 4), (-0.3, 7), (0.05, 1)):
        a = arr(run_graph(ours, [f"decimating_shift_addition_cc {rate} {dec}"], z), np.complex64)
        b = arr(run_graph(ref, [f"decimating_shift_addition_cc {rate} {dec}"], z), np.complex64)
        assert a.size == b.size and a.size > 0 and rel(a, b) < 1e-5, (rate, dec)


def test_wfm_graph_of_csdr_fm(clis):
    """The reference's canonical WFM receiver (csdr-fm:41, README.md:66) end to end:
    convert_u8_f | fmdemod_quadri_cf | fractional_decimator_ff 5 | deemphasis_wfm_ff 48000 50e-6 | convert_f_s16, plus limit_ff."""
    ours, ref = clis
    data = fm_u8(480_000, seed=11)
    stages = ["convert_u8_f", "fmdemod_quadri_cf", "fractional_decimator_ff 5", "deemphasis_wfm_ff 48000 50e-6", "limit_ff 0.5"]
    a = arr(run_graph(ours, stages, data), np.float32); b = arr(run_graph(ref, stages, data), np.float32)
    assert a.size == b.size and a.size > 90_000 and rel(a, b) < 1e-5
    a16 = arr(run_graph(ours, stages + ["convert_f_s16"], data), np.int16); b16 = arr(run_graph(ref, stages + ["convert_f_s16"], data), np.int16)
    assert a16.size == b16.size and np.abs(a16.astype(np.int32) - b16.astype(np.int32)).max() <= 1


def test_fft_commands(clis):
    ours, ref = clis
    rng = np.random.default_rng(7)
    z = (rng.uniform(-1, 1, 120_000) + 1j * rng.uniform(-1, 1, 120_000)).astype(np.complex64)
    for stages in (["bandpass_fir_fft_cc -0.05 0.05 0.002 HAMMING"], ["bandpass_fir_fft_cc 0.1 0.3 0.05"],
                   ["fastddc_fwd_cc 64 0.002", "fastddc_inv_cc 0.1 64 0.002"], ["fastddc_fwd_cc 8", "fastddc_inv_cc -0.21 8"]):
        a = arr(run_graph(ours, stages, z.tobytes()), np.complex64)
        b = arr(run_graph(ref, stages, z.tobytes()), np.complex64)
        assert a.size == b.size and a.size > 0, stages
        assert rel(a, b) < 1e-5, stages


def test_spectrum_and_unroll_commands(clis):
    ours, ref = clis
    rng = np.random.default_rng(12)
    z = (rng.uniform(-1, 1, 150_000) + 1j * rng.uniform(-1, 1, 150_000)).astype(np.complex64)
    a = arr(run_graph(ours, ["shift_unroll_cc 0.123"], z.tobytes()), np.complex64); b = arr(run_graph(ref, ["shift_unroll_cc 0.123"], z.tobytes()), np.complex64)
    assert a.size == b.size and rel(a, b) < 1e-6
    for stages in (["fft_cc 1024 1024 HAMMING", "logpower_cf -70"], ["fft_cc 2048 500", "logaveragepower_cf -70 2048 4"], ["fft_cc 512 3000 BLACKMAN"]):
        ra = run_graph(ours, stages, z.tobytes()); rb = run_graph(ref, stages, z.tobytes())
        assert len(ra) == len(rb) and len(ra) > 0, stages
        if stages[-1].startswith("fft_cc"):
            assert rel(arr(ra, np.complex64), arr(rb, np.complex64)) < 1e-5
        else:
            da, db = arr(ra, np.float32), arr(rb, np.float32)
            assert np.abs(da - db).max() < 5e-3, stages                              # dB values; FFT rounding differences on weak bins


def test_dynamic_bufsize_preamble(clis):
    ours, ref = clis
    z = np.random.default_rng(9).uniform(-1, 1, 2 * 70_000).astype(np.float32)
    head = b"csdr" + np.array([2048], np.int32).tobytes()
    env = {"CSDR_DYNAMIC_BUFSIZE_ON": "1"}
    stages = ["fir_decimate_cc 10 0.05 HAMMING", "fmdemod_quadri_cf"]
    a = run_graph(ours, stages, head + z.tobytes(), env); b = run_graph(ref, stages, head + z.tobytes(), env)
    assert a[:8] == b[:8] and len(a) == len(b)                       # the next-stage preamble is forwarded identically
    assert rel(arr(a[8:], np.float32), arr(b[8:], np.float32)) < 1e-5


def test_reference_binary_runs_on_our_library(clis):
    """Drop-in at the dynamic-link boundary: the reference's own csdr binary with libcsdr_b200.so preloaded computes its
    hot-path functions on the GPU (every other symbol still resolves to the reference library)."""
    ours, ref = clis
    if ref is REFERENCE:
        pytest.skip("needs the reference csdr binary itself (oracle/_ref/csdr_ref)")
    data = fm_u8(300_000, seed=3)
    stages = ["convert_u8_f", "fir_decimate_cc 10 0.05 HAMMING", "fmdemod_quadri_cf"]
    plain = arr(run_graph(ref, stages, data), np.float32)
    pre = arr(run_graph(ref, stages, data, env={"LD_PRELOAD": str(LIB), "CSDRB_TRACE": "1"}), np.float32)
    assert pre.size == plain.size and rel(pre, plain) < 1e-5
    assert not np.array_equal(pre, plain) or True                    # (sums are ordered differently on the GPU; equality is not required)
    # prove the preloaded library actually did the work: it counts its kernel launches and reports them at exit
    e = dict(os.environ); e.update({"LD_PRELOAD": str(LIB), "CSDRB_TRACE": "1"})
    r = subprocess.run(["bash", "-c", f"{ref} fir_decimate_cc 10 0.05 HAMMING"], input=np.zeros(2 * 40000, np.float32).tobytes(),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e, timeout=60)
    assert b"libcsdr_b200: " in r.stderr and b"kernel launches" in r.stderr, r.stderr[-500:]
