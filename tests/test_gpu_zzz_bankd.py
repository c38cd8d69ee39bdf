"""GPU tests (-m gpu) of csdr-bankd (csdr_b200/host/bankd.c, SURVEY 8(f) rank 2): one process turns one wideband u8/f32 IQ stream
(stdin or an nmux-style raw TCP stream) into per-channel NFM audio.  Per channel the stream must equal the README.md:87 graph run by
the oracle over the whole stream, whatever the daemon's block size."""
import os
import socket
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = Path(__file__).resolve().parent.parent
BANKD = ROOT / "csdr_b200" / "csdr-bankd"
GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_golden.npz")
RATES = (-0.41, -0.2, 0.03, 0.27, 0.44)
D, BW = 50, 0.005


@pytest.fixture(scope="module")
def bankd():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    from csdr_b200.build import build
    build()
    assert BANKD.exists()
    return str(BANKD)


def wideband_u8(n, seed=7):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    z = sum(0.17 * np.exp(1j * (2 * np.pi * (-r) * t + np.cumsum(2 * np.pi * 3000.0 / 2.4e6 * np.sin(2 * np.pi * (700.0 + 300 * k) / 2.4e6 * t))))
            for k, r in enumerate(RATES))
    z = z + 0.003 * (rng.normal(size=n) + 1j * rng.normal(size=n))
    iq = np.empty(2 * n); iq[0::2] = z.real; iq[1::2] = z.imag
    return np.clip(np.floor(iq * 127.5 + 128), 0, 255).astype(np.uint8)


def oracle_channel(oracle, wide_c64, rate, taps, tail):
    sh, _ = oracle.shift_addition_cc(wide_c64, float(np.float32(rate)), 0.0, 1024)
    d = oracle.fmdemod_quadri_cf(oracle.fir_decimate_cc(sh, D, taps))[0]
    if tail == "none":
        return d
    return oracle.convert_f_s16(oracle.fastagc_ff(oracle.deemphasis_nfm_ff(oracle.limit_ff(d, 1.0), GOLD["nfm_taps_48000"]), 1024, 1.0))


def MULTI_DEVICES():
    """device lists for the daemon's --devices mode: one device always; two when the box has them.  Counted as the daemon counts them: the CUDA
    runtime (csdrb_device_count) in a process of its own.  torch.cuda.device_count() takes NVML's count when NVML answers; on a machine whose
    NVML listed GPUs the process could not open, "--devices 0,1" failed with "invalid device ordinal" with one GPU usable."""
    r = subprocess.run([sys.executable, "-c", "import csdr_b200; print(csdr_b200.lib().csdrb_device_count())"], cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    out = r.stdout.split()
    assert r.returncode == 0 and out and out[-1].lstrip("-").isdigit(), ("csdrb_device_count", r.returncode, r.stdout, r.stderr[-500:])
    return ["0", "0,1"] if int(out[-1]) >= 2 else ["0"]


def stream_used(oracle, n, block):
    """samples of an n-sample stream the daemon processes: the first call takes `block`, every later one as many new samples as the previous call
    consumed (constant presented size, csdr.c:1172-1174); a partial last read is dropped"""
    T = oracle.firdes_filter_len(BW)
    consumed = ((block - T) // D + 1) * D
    return block + ((n - block) // consumed) * consumed if n >= block else 0


def run(bankd, args, data, sinks, timeout=300):
    cmd = [bankd] + args + [f"{r}:{p}" for r, p in zip(RATES, sinks)]
    r = subprocess.run(cmd, input=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stderr.decode()


@pytest.mark.parametrize("block", [262144, 100_000])
def test_nfm_bank_equals_the_readme_graph_per_channel(bankd, oracle, tmp_path, block):
    n = 6 * 262144
    u8 = wideband_u8(n)
    used = stream_used(oracle, n, block)
    sinks = [tmp_path / f"ch{k}.s16" for k in range(len(RATES))]
    run(bankd, ["--block", str(block)], u8.tobytes(), sinks)
    wide = oracle.convert_u8_f(u8[:2 * used]).view(np.complex64)
    taps = oracle.firdes_lowpass_f(oracle.firdes_filter_len(BW), 0.5 / D)
    for rate, path in zip(RATES, sinks):
        got = np.fromfile(path, np.int16)
        want = oracle_channel(oracle, wide, rate, taps, "nfm")
        assert got.size == want.size and got.size >= 25 * 1024, (rate, got.size, want.size)
        assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1, rate       # floats equal to ~1e-6 -> s16 within one count
    # --devices with the NFM tail: the channels' discriminator rows come back from their devices and go through the tail on the first one -- the same
    # kernels on the same numbers, so the audio must be the single-device run's, byte for byte
    if block == 100_000:
        devices = MULTI_DEVICES()[-1]                                  # two devices where the box (or the emulator) has them
        short = u8[:2 * 7 * block].tobytes()                           # seven blocks: enough for several AGC blocks of audio per channel
        ssinks = [tmp_path / f"s{k}.s16" for k in range(len(RATES))]
        msinks = [tmp_path / f"m{k}.s16" for k in range(len(RATES))]
        run(bankd, ["--block", str(block)], short, ssinks)
        run(bankd, ["--block", str(block), "--devices", devices], short, msinks)
        for a, b in zip(ssinks, msinks):
            assert a.stat().st_size >= 4 * 2 * 1024 and a.read_bytes() == b.read_bytes(), devices


def test_raw_discriminator_output_and_f32_input(bankd, oracle, tmp_path):
    n = 3 * 131072
    u8 = wideband_u8(n, seed=9)
    wide = oracle.convert_u8_f(u8).view(np.complex64)
    sinks = [tmp_path / f"ch{k}.f32" for k in range(len(RATES))]
    run(bankd, ["--tail", "none", "--f32", "--block", "131072"], wide.tobytes(), sinks)
    taps = oracle.firdes_lowpass_f(oracle.firdes_filter_len(BW), 0.5 / D)
    used = stream_used(oracle, n, 131072)
    from oracle.pyoracle import rel_rms
    for rate, path in zip(RATES, sinks):
        got = np.fromfile(path, np.float32)
        want = oracle_channel(oracle, wide[:used], rate, taps, "none")
        assert got.size == want.size and rel_rms(got, want) < 1e-5, (rate, got.size, want.size)
    # the same stream through the one-process multi-GPU bank (csdrb_multi_bank_*): on one device it must give the same bytes (no NCCL involved),
    # with u8 input converted on the host; MULTI_DEVICES lists what the box offers (the CPU tier pretends to have two)
    for devices in MULTI_DEVICES():
        msinks = [tmp_path / f"m{devices.replace(',', '_')}_{k}.f32" for k in range(len(RATES))]
        run(bankd, ["--tail", "none", "--u8", "--block", "131072", "--devices", devices], u8.tobytes(), msinks)
        for a, b in zip(sinks, msinks):
            assert a.read_bytes() == b.read_bytes(), devices


def test_tcp_ingest_and_tcp_sink(bankd, tmp_path):
    """--in HOST:PORT reads the raw stream an nmux server would send; a tcp:PORT sink serves one listener.  Same bytes as stdin/file."""
    n = 4 * 65536
    u8 = wideband_u8(n, seed=11).tobytes()
    files = [tmp_path / f"a{k}.s16" for k in range(len(RATES))]
    run(bankd, ["--block", "65536"], u8, files)

    srv = socket.socket(); srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1); srv.bind(("127.0.0.1", 0)); srv.listen(1)
    in_port = srv.getsockname()[1]
    probe = socket.socket(); probe.bind(("127.0.0.1", 0)); out_port = probe.getsockname()[1]; probe.close()

    def feed():
        conn, _ = srv.accept()
        conn.sendall(u8); conn.close()

    received = bytearray()

    def listen():
        import time
        for _ in range(900):                                              # the daemon opens its listener after creating the bank (CUDA start-up first)
            try:
                c = socket.create_connection(("127.0.0.1", out_port), timeout=1); break
            except OSError:
                time.sleep(0.1)
        else:
            return
        c.settimeout(60)
        while True:
            chunk = c.recv(1 << 16)
            if not chunk:
                break
            received.extend(chunk)

    t1 = threading.Thread(target=feed, daemon=True); t2 = threading.Thread(target=listen, daemon=True)
    t1.start(); t2.start()
    sinks = [f"tcp:{out_port}"] + [str(tmp_path / f"b{k}.s16") for k in range(1, len(RATES))]
    run(bankd, ["--block", "65536", "--in", f"127.0.0.1:{in_port}"], b"", sinks)
    t1.join(30); t2.join(30)
    assert bytes(received) == files[0].read_bytes() and len(received) > 0
    for k in range(1, len(RATES)):
        assert (tmp_path / f"b{k}.s16").read_bytes() == files[k].read_bytes()
