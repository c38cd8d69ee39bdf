"""GPU tests (-m gpu) of the CLI's run-time control channel (csdr.c:252-343: --fd <inherited descriptor> / --fifo <path>, one value per line):
the value that is waiting when the process starts selects the initial tuning, exactly as if it had been given on the command line -- for our CLI and
for the reference CLI alike.  Re-tuning in MID-STREAM is made deterministic by writing the control line while the program is blocked in the read of block k: both programs poll the
channel after writing a block, so the new value takes effect from block k+1 on -- test_midstream_retune_at_a_known_block.  The same bodies run in the CPU
tier on the emulated library (tests/test_cli_emulated.py).  File name sorts last: not yet run on hardware."""
import os
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_gpu_cli import arr, clis, rel, run_graph  # noqa: E402,F401
from reference_cli import recorded  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@recorded
def _with_fd(cli, args_before, args_after, line, data, timeout=120):
    """run `cli <args_before> --fd N <args_after>` with `line` already waiting in the pipe behind descriptor N"""
    r, w = os.pipe()
    os.write(w, line.encode())
    try:
        p = subprocess.run([cli] + args_before + ["--fd", str(r)] + args_after, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, pass_fds=(r,), timeout=timeout)
    finally:
        os.close(r); os.close(w)
    assert p.returncode == 0, p.stderr[-1000:]
    return p.stdout


@recorded
def _with_fifo(cli, args_before, args_after, line, data, tmp_path, timeout=120):
    """the same through a named FIFO: the CLI blocks in open() until a writer shows up"""
    path = tmp_path / f"ctl_{abs(hash((cli, tuple(args_before), line))) % 10**8}"
    os.mkfifo(path)
    keep = []

    def writer():
        fd = os.open(path, os.O_WRONLY)
        os.write(fd, line.encode())
        keep.append(fd)                                                  # stay open until the CLI is done (a closed FIFO still reads as "no data")

    t = threading.Thread(target=writer, daemon=True); t.start()
    try:
        p = subprocess.run([cli] + args_before + ["--fifo", str(path)] + args_after, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout)
    finally:
        t.join(10)
        for fd in keep:
            os.close(fd)
    assert p.returncode == 0, p.stderr[-1000:]
    return p.stdout


def test_initial_tuning_through_the_control_channel(clis, tmp_path):
    ours, ref = clis
    rng = np.random.default_rng(12)
    z = (rng.uniform(-1, 1, 70_000) + 1j * rng.uniform(-1, 1, 70_000)).astype(np.complex64).tobytes()
    for cli in (ours, ref):
        plain = run_graph(cli, ["shift_addition_cc -0.085"], z)
        assert _with_fd(cli, ["shift_addition_cc"], [], "-0.085\n", z) == plain
        assert _with_fifo(cli, ["shift_addition_cc"], [], "-0.085\n", z, tmp_path) == plain
        assert _with_fd(cli, ["shift_unroll_cc"], [], "0.2\n", z) == run_graph(cli, ["shift_unroll_cc 0.2"], z)
        assert _with_fd(cli, ["bandpass_fir_fft_cc"], ["0.05"], "-0.1 0.2\n", z) == run_graph(cli, ["bandpass_fir_fft_cc -0.1 0.2 0.05"], z)
    # and the two programs agree with each other on the controlled runs
    a = arr(_with_fd(ours, ["shift_addition_cc"], [], "0.3\n", z), np.complex64)
    b = arr(_with_fd(ref, ["shift_addition_cc"], [], "0.3\n", z), np.complex64)
    assert a.size == b.size and rel(a, b) < 1e-5
    spectra_ours = run_graph(ours, ["fastddc_fwd_cc 8"], z); spectra_ref = run_graph(ref, ["fastddc_fwd_cc 8"], z)
    a = arr(_with_fd(ours, ["fastddc_inv_cc"], ["8"], "-0.21\n", spectra_ours), np.complex64)
    b = arr(_with_fd(ref, ["fastddc_inv_cc"], ["8"], "-0.21\n", spectra_ref), np.complex64)
    assert a.size == b.size and a.size > 0 and rel(a, b) < 1e-5


@recorded
def _retune_run(cli, args_before, args_after, first, second, blocks, out_block_bytes, retune_after, timeout=400):
    """Feed `blocks` one by one; the line `second` is written to the control descriptor while the program waits for block `retune_after`, i.e. after it has
    flushed block retune_after - 1 (a reader thread drains stdout; we wait until those bytes are there).  Both CLIs poll right after writing a block
    (csdr.c:920 / our poll_control), so the new tuning applies to every block after `retune_after` -- deterministically."""
    import time
    r, w = os.pipe()
    os.write(w, first.encode())
    p = subprocess.Popen([cli] + args_before + ["--fd", str(r)] + args_after, stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, pass_fds=(r,))
    got = bytearray()

    def drain():
        while True:
            chunk = p.stdout.read1(65536)                                 # whatever has arrived (read() would wait for 64 KiB: blocks can be tiny)
            if not chunk:
                return
            got.extend(chunk)

    t = threading.Thread(target=drain, daemon=True); t.start()
    try:
        for k, b in enumerate(blocks):
            if k == retune_after:
                deadline = time.time() + timeout                          # block k-1 has been flushed: the poll that followed its write is over
                while len(got) < retune_after * out_block_bytes:
                    assert time.time() < deadline and p.poll() is None, "the CLI did not deliver the blocks before the retune"
                    time.sleep(0.01)
                os.write(w, second.encode())                               # waiting in the pipe before block k's bytes arrive
            p.stdin.write(b); p.stdin.flush()
        p.stdin.close()
        assert p.wait(timeout=timeout) == 0
        t.join(timeout)
    finally:
        os.close(r); os.close(w)
        if p.poll() is None:
            p.kill()
    return bytes(got)


def test_midstream_retune_at_a_known_block(clis, oracle):
    """shift_addition_cc, bandpass_fir_fft_cc and fastddc_inv_cc retuned between two known blocks (csdr.c:289-323, :920): ours and the reference's CLI must
    produce the same stream, and for the NCO it must be the oracle's chain with the rate switched at that block and the phase carried through."""
    ours, ref = clis
    rng = np.random.default_rng(13)
    B = 16384                                                             # shift_addition_cc reads 16384-sample blocks (csdr.c:189-190)
    nb, k0 = 4, 2
    z = (rng.uniform(-1, 1, nb * B) + 1j * rng.uniform(-1, 1, nb * B)).astype(np.complex64)
    blocks = [z[k * B:(k + 1) * B].tobytes() for k in range(nb)]
    outs = {}
    for cli in (ours, ref):
        outs[cli] = arr(_retune_run(cli, ["shift_addition_cc"], [], "0.11\n", "-0.23\n", blocks, B * 8, k0), np.complex64)
        assert outs[cli].size == nb * B
    # the oracle's chain: rate 0.11 for blocks 0..k0, then -0.23, the phase continuing (the CLI re-runs shift_addition_init, not the phase)
    a, ph = oracle.shift_addition_cc(z[:(k0 + 1) * B], 0.11, 0.0, 1024)
    b, _ = oracle.shift_addition_cc(z[(k0 + 1) * B:], -0.23, float(ph), 1024)
    want = np.concatenate([a, b])
    for cli in (ours, ref):
        e = rel(outs[cli], want)
        assert e < 1e-5, (cli, e)
    e = rel(outs[ours], outs[ref])
    assert e < 1e-5, f"ours vs reference CLI after a mid-stream retune: rel-RMS {e:.3e}"
    # bandpass_fir_fft_cc: blocks of input_size samples; new band edges from block k0+1 on
    T = oracle.firdes_filter_len(0.05)
    N = 1
    while N < T:
        N <<= 1
    if N - T < 200:
        N <<= 1
    isz = N - T + 1
    zb = z[:8 * isz]
    bl = [zb[k * isz:(k + 1) * isz].tobytes() for k in range(8)]
    o = [arr(_retune_run(cli, ["bandpass_fir_fft_cc"], ["0.05"], "-0.1 0.2\n", "0.05 0.3\n", bl, isz * 8, 4), np.complex64) for cli in (ours, ref)]
    assert o[0].size == o[1].size and o[0].size >= 8 * isz
    e = rel(o[0][:8 * isz], o[1][:8 * isz])
    assert e < 1e-5, f"bandpass_fir_fft_cc retuned mid-stream: rel-RMS {e:.3e}"
    static = arr(run_graph(ours, ["bandpass_fir_fft_cc -0.1 0.2 0.05"], zb.tobytes()), np.complex64)
    assert rel(o[0][:4 * isz], static[:4 * isz]) < 1e-6 and rel(o[0][6 * isz:8 * isz], static[6 * isz:8 * isz]) > 0.05      # the retune really happened
