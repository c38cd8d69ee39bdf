"""GPU parity tests (-m gpu) for the IMA ADPCM encoder of SURVEY 8(f) rank 4 (ima_adpcm.c:95-150, csdr.c:1739-1767, 1891-1904): bank rows, drop-in,
CLI commands against the reference CLI.  (File name sorts last on purpose: written after the round's GPU budget was spent; so far executed only under
the CPU tier's emulator, tests/test_kernels_emulated.py::test_ima_adpcm_rows_bit_exact and the emulated CLI.)"""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_gpu_cli import arr, clis, run_graph  # noqa: E402,F401

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import csdr_b200
    csdr_b200.lib()
    return csdr_b200


def test_adpcm_rows_and_waterfall_lines_bit_exact(gpu, oracle):
    rng = np.random.default_rng(4)
    rows, n = 300, 2050
    x = (rng.standard_normal((rows, n)) * rng.choice([10, 300, 5000, 40000], (rows, 1))).clip(-32768, 32767).astype(np.int16)
    out, st = gpu.encode_ima_adpcm_rows_i16_u8(torch.from_numpy(x).cuda())
    out = out.cpu().numpy(); st = st.cpu().numpy()
    for r in range(0, rows, 7):
        want, (wi, wp) = oracle.encode_ima_adpcm_i16_u8(x[r])
        assert np.array_equal(out[r], want) and (st[r, 0], st[r, 1]) == (wi, wp), r
    for fft_size in (16, 511, 2048):
        db = rng.uniform(-130, 10, (rows, fft_size)).astype(np.float32); db[0, :3] = [np.nan, 400.0, -400.0]
        got = gpu.compress_fft_adpcm_rows_f_u8(torch.from_numpy(db).cuda()).cpu().numpy()
        assert np.array_equal(got, oracle.compress_fft_adpcm_f_u8(db, fft_size)), fft_size
    y, st = gpu.libcsdr.encode_ima_adpcm_i16_u8(x[0], 5, 1000)
    want, wst = oracle.encode_ima_adpcm_i16_u8(x[0], 5, 1000)
    assert np.array_equal(y, want) and st == wst


def test_adpcm_commands(clis):
    """compress_fft_adpcm_f_u8 (one fresh encoder per waterfall line) and encode_ima_adpcm_i16_u8 (state carried) -- byte for byte"""
    ours, ref = clis
    rng = np.random.default_rng(6)
    db = rng.uniform(-120, -20, 9 * 1024).astype(np.float32).tobytes()
    assert run_graph(ours, ["compress_fft_adpcm_f_u8 1024"], db) == run_graph(ref, ["compress_fft_adpcm_f_u8 1024"], db)
    pcm = (rng.standard_normal(20_000) * 3000).clip(-32768, 32767).astype(np.int16).tobytes()
    for name in ("encode_ima_adpcm_i16_u8", "encode_ima_adpcm_s16_u8"):
        assert run_graph(ours, [name], pcm) == run_graph(ref, [name], pcm)


def test_openwebrx_waterfall_chain(clis):
    """fft_cc | logaveragepower_cf | fft_exchange_sides_ff | compress_fft_adpcm_f_u8 (the OpenWebRX waterfall): same framing as the reference CLI;
    the dB values agree to 2e-5 dB, so after *100 and truncation a few centi-dB steps may differ -- the compressed lines must agree almost everywhere."""
    ours, ref = clis
    rng = np.random.default_rng(8)
    n = 1024 * 64
    t = np.arange(n)
    z = (0.5 * np.exp(2j * np.pi * 0.11 * t) + 0.05 * (rng.normal(size=n) + 1j * rng.normal(size=n))).astype(np.complex64).tobytes()
    half = np.arange(4096, dtype=np.float32).tobytes()
    assert run_graph(ours, ["fft_exchange_sides_ff 1024"], half) == run_graph(ref, ["fft_exchange_sides_ff 1024"], half)
    stages = ["fft_cc 1024 2048", "logaveragepower_cf -70 1024 4", "fft_exchange_sides_ff 1024", "compress_fft_adpcm_f_u8 1024"]
    a = arr(run_graph(ours, stages, z), np.uint8); b = arr(run_graph(ref, stages, z), np.uint8)
    assert a.size == b.size and a.size >= 4 * 517
    assert np.mean(a == b) > 0.95                                          # a centi-dB step that flips perturbs the next few ADPCM nibbles
