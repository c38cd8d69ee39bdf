"""GPU parity tests (-m gpu) for shift_math_cc (SURVEY 8(f) rank 3; libcsdr.c:186-209): drop-in, bank, CLI command against the reference CLI.
(File name sorts last on purpose: this kernel was written after the round's GPU budget was spent and has only run under the CPU tier's
emulator, tests/test_kernels_emulated.py::test_shift_math_bank.)"""
from pathlib import Path

import sys

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_gpu_cli import arr, clis, rel, run_graph  # noqa: E402,F401  (the CLI suite's fixture and helpers)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_golden.npz")


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    import csdr_b200
    csdr_b200.lib()
    return csdr_b200


def _rel(y, ref):
    from oracle.pyoracle import rel_rms
    return rel_rms(y, ref)


def test_shift_math_dropin_and_bank(gpu, oracle):
    y, ph = gpu.libcsdr.shift_math_cc(GOLD["shift_in"], -0.085, -7.5, 1024)
    assert np.float32(ph) == GOLD["math_phase"] and _rel(y, GOLD["math_out"]) < 1e-6
    rng = np.random.default_rng(3)
    rates = np.array([-0.5, -0.31, -0.085, 0.0, 1e-4, 0.2, 0.4999, 0.5], np.float32)
    ph0 = np.array([0.0, 3.0, -7.5, 100.0, 6.2831855, 1.0, 2.0, -0.0], np.float32)
    for n in (1, 255, 257, 10_001, 300_000):
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        out, ph = gpu.shift_math_bank_cc(torch.from_numpy(x).cuda(), rates, phases=torch.from_numpy(ph0).cuda())
        out = out.cpu().numpy(); ph = ph.cpu().numpy()
        for c, r in enumerate(rates):
            want, wph = oracle.shift_math_cc(x, float(r), float(ph0[c]))
            assert np.float32(wph).view(np.uint32) == ph[c].view(np.uint32), (n, c)
            assert _rel(out[c], want) < 1e-7, (n, c)


def test_shift_math_command(clis):
    """csdr.c:703-718 against the unmodified reference CLI (1024-sample calls, phase carried from call to call)"""
    ours, ref = clis
    z = (np.random.default_rng(3).uniform(-1, 1, 50_000) + 1j * np.random.default_rng(4).uniform(-1, 1, 50_000)).astype(np.complex64).tobytes()
    for rate in (0.2, -0.085, 0.4999):
        a = arr(run_graph(ours, [f"shift_math_cc {rate}"], z), np.complex64)
        b = arr(run_graph(ref, [f"shift_math_cc {rate}"], z), np.complex64)
        assert a.size == b.size and a.size > 0 and rel(a, b) < 1e-6, rate
