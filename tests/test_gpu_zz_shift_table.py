"""GPU parity tests (-m gpu) for shift_table_cc (SURVEY 8(f) rank 3; libcsdr.c:210-260): bank, drop-in, CLI command against the reference CLI.
The index arithmetic is pinned to the reference's own build (oracle.c), so with the same table the samples are identical.
(File name sorts last: written after the round's GPU budget was spent; executed so far only under the CPU tier's emulator.)"""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_gpu_cli import arr, clis, rel, run_graph  # noqa: E402,F401

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import csdr_b200
    csdr_b200.lib()
    return csdr_b200


def test_shift_table_bank_and_dropin_bit_exact(gpu, oracle):
    rng = np.random.default_rng(21)
    rates = np.array([-0.5, -0.31, -0.085, 0.0, 1e-4, 0.2, 0.4999, 0.5], np.float32)
    ph0 = np.array([0.0, 3.0, 1.5707964, 6.2831855, 0.5, 1.0, 2.0, 4.7], np.float32)
    for n, size in ((257, 65536), (10_001, 65536), (200_000, 65536), (20_000, 1024)):
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        table = oracle.shift_table_init(size)
        out, ph = gpu.shift_table_bank_cc(torch.from_numpy(x).cuda(), rates, table, phases=torch.from_numpy(ph0).cuda())
        out = out.cpu().numpy(); ph = ph.cpu().numpy()
        for c, r in enumerate(rates):
            want, wph, _bad = oracle.shift_table_cc(x, float(r), table, float(ph0[c]))
            assert np.float32(wph).view(np.uint32) == ph[c].view(np.uint32), (n, c)
            assert np.array_equal(out[c], want), (n, size, c, int(np.sum(out[c] != want)))
    x = (rng.uniform(-1, 1, 40_000) + 1j * rng.uniform(-1, 1, 40_000)).astype(np.complex64)
    table = gpu.libcsdr.shift_table_init(65536)
    assert np.abs(table - oracle.shift_table_init(65536)).max() == 0                # host table: the same expression as the oracle's
    y, ph = gpu.libcsdr.shift_table_cc(x, -0.085, table, 0.3, 16384)
    want, wph, _ = oracle.shift_table_cc(x, -0.085, table, 0.3, 16384)
    assert np.array_equal(y, want) and np.float32(ph) == np.float32(wph)


def test_shift_table_command(clis):
    """csdr.c:725-747 against the unmodified reference CLI.  The two programs build their tables with different sin() implementations (the reference
    build's is libmvec's), one ulp apart for some entries, so the comparison is to 1e-6, not to the bit."""
    ours, ref = clis
    z = (np.random.default_rng(3).uniform(-1, 1, 100_000) + 1j * np.random.default_rng(4).uniform(-1, 1, 100_000)).astype(np.complex64).tobytes()
    for args in ("0.2", "-0.085", "0.4999 1024"):
        a = arr(run_graph(ours, [f"shift_table_cc {args}"], z), np.complex64)
        b = arr(run_graph(ref, [f"shift_table_cc {args}"], z), np.complex64)
        assert a.size == b.size and a.size > 0 and rel(a, b) < 1e-6, args
