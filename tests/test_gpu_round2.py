"""GPU parity tests added in round 2 (run with -m gpu on the B200 box), all through the C ABI of libcsdr_b200.so:
  * the u8 front end fused into the FIR bank (convert_u8_f | fir_decimate_cc, csdr-fm:41), device and host (end-to-end) calls;
  * the table-driven phase chains (csrc/phase_table.cuh): long chains, every rate class, bit-exact carried phases vs the oracle's loops;
  * the fold-based fastddc inverse bank on ragged channel / block counts, against the round-1 kernels and the oracle;
  * config 2 against the COMPILED reference on 8 channels x 262 144 samples (SURVEY 8(d)) and every 32nd channel of the full-size bank;
  * a retune of the streaming DDC bank in the middle of an NCO chunk: the phase stays continuous (ADVICE r1).
Every tolerance assert prints the value it achieved.
"""
import os
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
REF = np.load(Path(__file__).parent / "golden" / "ref_outputs.npz")         # the compiled reference on the seeded inputs below (make_ref_outputs.py)
TOL = 1e-5                                                              # BASELINE.json north_star: 1e-5 relative RMS for float blocks


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device; refusing to fall back to anything else")
    import csdr_b200
    csdr_b200.lib()
    return csdr_b200


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cplx(rng, *shape, amp=1.0):
    return ((rng.uniform(-1, 1, shape) + 1j * rng.uniform(-1, 1, shape)) * amp).astype(np.complex64)


def _at(y, key):
    """(y at the positions where the reference's output is stored, the stored values); the lengths must match"""
    from oracle.pyoracle import pick_idx
    n, want = int(REF[key + "_n"]), REF[key]
    assert y.size == n, (key, y.size, n)
    return y[pick_idx(n, want.size)], want


def _rel(y, ref):
    from oracle.pyoracle import rel_rms
    return rel_rms(y, ref)


# ------------------------------------------------------------------------------------------ u8 front end
@pytest.mark.parametrize("D,T,n", [(10, 199, 262_144 + 3), (10, 79, 16_384), (50, 801, 100_003), (10, 199, 8321), (7, 33, 5000)])
def test_u8_fir_bank_equals_convert_then_filter(gpu, oracle, D, T, n):
    rng = np.random.default_rng(n)
    ch = 5
    stride = (n + 7) & ~7
    u8 = rng.integers(0, 256, (ch, stride, 2), dtype=np.uint8)
    u8[0, :256, 0] = np.arange(256); u8[0, :256, 1] = np.arange(255, -1, -1)
    taps = oracle.firdes_lowpass_f(T, 0.5 / D)
    d8 = _dev(u8)[:, :n]                                                  # rows padded to a multiple of 8 samples (16-byte row starts): the fused path
    y = gpu.fir_decimate_bank_u8_cc(d8, D, taps).cpu().numpy()
    f = gpu.convert_u8_f(_dev(u8.reshape(ch, -1)))                        # the padded rows: an even row stride keeps the cf32 bank on the same (fast) kernel
    assert np.array_equal(f.cpu().numpy()[0, : 2 * n], oracle.convert_u8_f(u8[0, :n].reshape(-1)))
    y2 = gpu.fir_decimate_bank_cc(f.view(ch, stride, 2)[:, :n], D, taps).cpu().numpy()
    if (D, T) != (7, 33):
        assert np.array_equal(y, y2), "fused u8 path must equal convert_u8_f followed by the cf32 bank bit for bit"
    worst = 0.0
    for c in range(ch):
        xc = oracle.convert_u8_f(u8[c, :n].reshape(-1)).view(np.complex64)
        e = _rel(y[c], oracle.fir_decimate_cc(xc, D, taps)); worst = max(worst, e)
        assert e < TOL, f"channel {c}: rel-RMS {e:.3e} (bar {TOL})"
    print(f"u8 FIR bank D={D} T={T}: worst rel-RMS {worst:.2e}")
    # rows that do NOT start on 16-byte boundaries: the two-launch path behind the same entry point
    odd = _dev(u8.reshape(ch, -1)[:, : 2 * (n - 3)].copy().reshape(ch, n - 3, 2))
    if (n - 3) % 8:
        y3 = gpu.fir_decimate_bank_u8_cc(odd, D, taps).cpu().numpy()
        xc = oracle.convert_u8_f(u8[1, : n - 3].reshape(-1)).view(np.complex64)
        e = _rel(y3[1], oracle.fir_decimate_cc(xc, D, taps))
        assert e < TOL, f"unaligned rows: rel-RMS {e:.3e}"


def test_u8_host_call_end_to_end(gpu, oracle):
    rng = np.random.default_rng(5)
    ch, n, D, T = 12, 300_000, 10, 199
    taps = oracle.firdes_lowpass_f(T, 0.5 / D)
    h = gpu.PinnedArray((ch, n, 2), np.uint8)
    h.array[:] = rng.integers(0, 256, (ch, n, 2), dtype=np.uint8)
    out = gpu.fir_decimate_bank_u8_host(h.array, D, taps, chunk_channels=5)          # 3 chunks: 5 + 5 + 2 channels through the 3-stream pipeline
    for c in (0, 4, 5, 11):
        xc = oracle.convert_u8_f(h.array[c].reshape(-1)).view(np.complex64)
        e = _rel(out[c], oracle.fir_decimate_cc(xc, D, taps))
        assert e < TOL, f"channel {c}: rel-RMS {e:.3e}"
    h.close()


# ------------------------------------------------------------------------------------------ phase chains on the wrap table
@pytest.mark.parametrize("chunk,nchunks", [(1024, 300), (64, 1500), (1000, 130), (4096, 100)])
def test_long_phase_chains_are_bit_exact(gpu, oracle, chunk, nchunks):
    """> 96 chunks per call: the chain kernels run on the register-resident wrap table (csrc/phase_table.cuh).  The carried phase must be the
    very float the reference's `while` loops leave (libcsdr_gpl.c:48-50) for slow, fast, negative and tiny rates alike."""
    n = chunk * nchunks + 17
    rates = np.array([-0.4999, -0.41, -0.25, -0.085, -1e-3, 0.0, 1e-4, 0.0123, 0.2, 0.3333, 0.45, 0.4999], np.float32)
    x = _dev(_cplx(np.random.default_rng(chunk), n))
    ph0 = np.random.default_rng(1).uniform(-3.1, 3.1, rates.size).astype(np.float32)
    y, ph = gpu.shift_addition_bank_cc(x, rates, phases=_dev(ph0), chunk=chunk)
    ph = ph.cpu().numpy()
    xh = x.cpu().numpy()
    for c, r in enumerate(rates):
        want, wph = oracle.shift_addition_cc(xh, float(r), float(ph0[c]), chunk)
        assert np.float32(wph) == np.float32(ph[c]), f"rate {r}: carried phase {ph[c]!r} vs reference {wph!r}"
        e = _rel(y[c].cpu().numpy(), want)
        assert e < 2e-6, f"rate {r}: rel-RMS {e:.3e}"


# ------------------------------------------------------------------------------------------ fastddc inverse plan (look-ahead) == stateless bank
@pytest.mark.parametrize("channels,nblocks", [(5, 7), (64, 256)])
def test_fastddc_inverse_plan_equals_the_stateless_bank(gpu, oracle, channels, nblocks):
    """csdrb_fastddc_inv_plan_* prepares run k+1 (state chain + phasors) on its own stream during run k: outputs, counts and carried state must be those
    of csdrb_fastddc_inv_bank_cc BIT FOR BIT over six runs with a retune in the middle; BASELINE config 3's size is the second case."""
    import torch
    bw, dec, runs = 0.002, 64, 6
    ddc = gpu.fastddc_init(bw, dec, 0.0)
    rng = np.random.default_rng(channels)
    shifts = list(np.linspace(-0.43, 0.41, channels))
    plan = gpu.FastddcInvPlan(shifts, dec, bw, nblocks)
    st = None; ov = None
    try:
        for r in range(runs):
            x = _dev(_cplx(rng, nblocks * ddc.input_size, amp=0.5))
            sp, ov = gpu.fastddc_fwd_cc(x, ddc, overlap=ov)
            if r == 3:                                                  # retune one channel in both
                c, new = channels // 2, 0.2345
                plan.set_shift(c, new)
                shifts[c] = new
                d = gpu.fastddc_init(bw, dec, new)
                st["taps_fft"][c].copy_(gpu.fastddc_make_taps_fft(d, new, dec, "HAMMING", "cuda"))
                row = torch.from_numpy(gpu._fastddc_chan_rows([d])[0]).cuda()
                st["chan"][c].copy_(row)
            want, wc, st = gpu.fastddc_inv_bank_cc(sp, shifts, dec, bw, state=st)
            got, gc = plan.run(sp)
            torch.cuda.synchronize()
            assert torch.equal(gc, wc), f"run {r}: counts differ"
            n = int(wc.max())
            live = (torch.arange(n, device="cuda")[None, :] < wc[:, None])[..., None]                 # beyond a channel's count the buffers hold whatever they held
            a = torch.view_as_real(got[:, :n]).view(torch.int32) * live, torch.view_as_real(want[:, :n]).view(torch.int32) * live
            assert torch.equal(*a), f"run {r}: outputs differ"
        remain, phase = plan.state()
        assert np.array_equal(remain, st["remain"].cpu().numpy()) and np.array_equal(phase.view(np.uint32), st["phase"].cpu().numpy().view(np.uint32))
    finally:
        plan.close()


# ------------------------------------------------------------------------------------------ fastddc inverse: fold path vs round-1 kernels vs oracle
@pytest.mark.parametrize("channels,nblocks", [(1, 1), (3, 5), (17, 33), (20, 130)])
def test_fastddc_fold_path_ragged_banks(gpu, oracle, channels, nblocks):
    bw, dec = 0.002, 64
    ddc = gpu.fastddc_init(bw, dec, 0.0)
    rng = np.random.default_rng(channels * 1000 + nblocks)
    x = _cplx(rng, nblocks * ddc.input_size, amp=0.5)
    shifts = list(np.linspace(-0.43, 0.41, channels))
    sp, _ = gpu.fastddc_fwd_cc(_dev(x), ddc)
    out, counts, st = gpu.fastddc_inv_bank_cc(sp, shifts, dec, bw)
    out = out.cpu().numpy(); counts = counts.cpu().numpy()
    o_ddc, _ = oracle.fastddc_init(bw, dec, 0.0)
    want_sp = oracle.fastddc_fwd(x, o_ddc)
    worst = 0.0
    for c in sorted({0, channels // 2, channels - 1}):
        want = oracle.fastddc_inv(want_sp, bw, dec, shifts[c])
        assert counts[c] == want.size
        e = _rel(out[c, :want.size], want); worst = max(worst, e)
        assert e < TOL / 2, f"channel {c}: rel-RMS {e:.3e}"
    print(f"fastddc fold path {channels} ch x {nblocks} blocks: worst rel-RMS {worst:.2e}")
    # state carried into a second call (remain / phase chain incl. the wrap table for nblocks > 96)
    x2 = _cplx(rng, 3 * ddc.input_size, amp=0.5)
    sp_all, _ = gpu.fastddc_fwd_cc(_dev(np.concatenate([x, x2])), ddc)
    out2, counts2, _ = gpu.fastddc_inv_bank_cc(sp_all[nblocks:].contiguous(), shifts, dec, bw, state=st)
    c = channels - 1
    want_all = oracle.fastddc_inv(oracle.fastddc_fwd(np.concatenate([x, x2]), o_ddc), bw, dec, shifts[c])
    got = np.concatenate([out[c, :counts[c]], out2[c, :int(counts2[c])].cpu().numpy()])
    e = _rel(got, want_all)
    assert got.size == want_all.size and e < TOL / 2, f"streamed: rel-RMS {e:.3e}"


# ------------------------------------------------------------------------------------------ config 2 vs the compiled reference
def test_config2_against_compiled_reference_8x262144(gpu):
    """SURVEY 8(d): config 2 checked against the unmodified reference build on >= 8 channels x the first 262 144 samples
    (its outputs at 512 seeded positions per channel, tests/golden/ref_outputs.npz)."""
    T, D, C, N = 199, 10, 8, 262_144
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    x = np.stack([_cplx(np.random.default_rng(100 + c), N) for c in range(C)])
    y = gpu.fir_decimate_bank_cc(_dev(x), D, taps).cpu().numpy()
    worst = 0.0
    for c in range(C):
        e = _rel(*_at(y[c], f"cfg2_ch{c}")); worst = max(worst, e)
        assert e < TOL, f"channel {c}: rel-RMS {e:.3e} vs the compiled reference (bar {TOL})"
    print(f"config 2 vs the reference build, 8 ch x 262144: worst rel-RMS {worst:.2e}")


def test_config2_full_size_every_32nd_channel(gpu, oracle):
    """the 256 x 2.4 M bank of the bench: every 32nd channel's first 120 000 outputs against the oracle (the whole channel would take minutes on the CPU)"""
    T, D, C, N = 199, 10, 256, 2_400_000
    taps = gpu.firdes_lowpass_f(T, 0.5 / D)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.rand((C, N, 2), generator=g, device="cuda") * 2 - 1
    y = gpu.fir_decimate_bank_cc(x, D, taps)
    head = 120_000 * D + T
    worst = 0.0
    for c in range(0, C, 32):
        xc = x[c, :head].cpu().numpy().view(np.complex64).reshape(-1)
        want = oracle.fir_decimate_cc(xc, D, taps)[:120_000]
        e = _rel(y[c, :120_000].cpu().numpy(), want); worst = max(worst, e)
        assert e < TOL, f"channel {c}: rel-RMS {e:.3e}"
    print(f"config 2 full size, every 32nd channel: worst rel-RMS {worst:.2e}")


# ------------------------------------------------------------------------------------------ retune in the middle of an NCO chunk
def test_ddc_bank_retune_keeps_the_phase_continuous(gpu, oracle):
    """csdrb_ddc_bank_set_rate between two blocks whose boundary falls inside a 1024-sample NCO chunk: the bank closes the chunk at the retune sample
    (a shorter shift_addition_cc call) and continues from the phase AT that sample, so the stream equals the reference chain cut the same way."""
    D, bw = 50, 0.005
    T = oracle.firdes_filter_len(bw)
    taps = oracle.firdes_lowpass_f(T, 0.5 / D)
    rng = np.random.default_rng(3)
    n1 = 20_000
    rates = np.array([0.1, -0.2, 0.31], np.float32)
    x = _cplx(rng, 60_000, amp=0.5)
    bank = gpu.DdcBank(rates, D, taps, demod=False, chunk=1024)
    o1 = bank.process(_dev(x[:n1])).cpu().numpy()
    used = o1.shape[1] * D
    assert used % 1024 != 0 and bank.offset == used % 1024               # the retune will land inside a chunk
    bank.set_rate(1, 0.05)
    o2 = bank.process(_dev(x[used:used + 30_000])).cpu().numpy()
    assert bank.offset == (o2.shape[1] * D) % 1024                       # a fresh chunk started at the retune sample
    bank.close()
    for c, (r_old, r_new) in enumerate(zip([0.1, -0.2, 0.31], [0.1, 0.05, 0.31])):
        # reference chain: chunks of 1024 up to `used` (the last one shorter), then chunks of 1024 again with the new rate, phase carried through
        sh1, ph = oracle.shift_addition_cc(x[:used], r_old, 0.0, 1024)
        want1 = oracle.fir_decimate_cc(oracle.shift_addition_cc(x[:n1], r_old, 0.0, 1024)[0], D, taps)
        e1 = _rel(o1[c], want1)
        assert e1 < 2e-6, f"channel {c} before the retune: rel-RMS {e1:.3e}"
        sh2, _ = oracle.shift_addition_cc(x[used:used + 30_000], r_new, float(ph), 1024)
        want2 = oracle.fir_decimate_cc(sh2, D, taps)
        e2 = _rel(o2[c], want2)
        assert e2 < 2e-6, f"channel {c} after the retune: rel-RMS {e2:.3e} (a phase jump at the retune sample would show as O(1))"


# ------------------------------------------------------------------------------------------ one process, several GPUs (csdrb_multi_bank_*)
def test_multi_gpu_bank_equals_the_single_gpu_bank(gpu, oracle):
    """The sharded bank against the unsharded one (VERDICT r1: no multi-GPU parity on GPUs): contiguous channel slices per device, the wideband block
    broadcast with NCCL from device 0, two blocks in flight.  One device always (no NCCL involved); two when the box has them."""
    D, bw = 50, 0.005
    T = oracle.firdes_filter_len(bw)
    taps = oracle.firdes_lowpass_f(T, 0.5 / D)
    Cn, N, NB = 24, 200_000, 4
    rates = np.linspace(-0.44, 0.43, Cn).astype(np.float32)
    rng = np.random.default_rng(21)
    n_out = (N - T) // D + 1
    adv = n_out * D
    stream = _cplx(rng, adv * (NB - 1) + N, amp=0.4)
    ref_bank = gpu.DdcBank(rates, D, taps, demod=True, chunk=1024)
    want = np.concatenate([ref_bank.process(_dev(stream[k * adv:k * adv + N])).cpu().numpy() for k in range(NB)], axis=1)
    ref_bank.close()
    device_sets = [[0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in device_sets:
        mb = gpu.MultiBank(devs, rates, D, taps, demod=True, chunk=1024, max_block=N)
        assert sum(n for _, _, n in mb.slices()) == Cn and [d for d, _, _ in mb.slices()] == devs
        wide = [gpu.PinnedArray((N,), np.complex64) for _ in range(2)]
        outs = [gpu.PinnedArray((Cn, n_out), np.float32) for _ in range(NB)]
        tickets = []
        for k in range(NB):
            if k >= 2:
                assert mb.collect(tickets[k - 2]) == n_out             # frees wide[k & 1]
            wide[k & 1].array[:] = stream[k * adv:k * adv + N]
            tickets.append(mb.submit(wide[k & 1].array, outs[k].array))
        for t in tickets[-2:]:
            assert mb.collect(t) == n_out
        got = np.concatenate([o.array for o in outs], axis=1)
        assert np.array_equal(got, want), f"devices {devs}: sharded bank differs from the unsharded one"
        mb.close()
        [w.close() for w in wide]; [o.close() for o in outs]
    # one channel against the reference chain itself
    c = 5
    sh, _ = oracle.shift_addition_cc(stream, float(rates[c]), 0.0, 1024)
    ref = oracle.fmdemod_quadri_cf(oracle.fir_decimate_cc(sh, D, taps))[0][:want.shape[1]]
    e = _rel(want[c], ref)
    assert e < TOL, f"rel-RMS {e:.3e}"


# ------------------------------------------------------------------------------------------ fastagc_ff | convert_f_s16 fused
@pytest.mark.parametrize("block", [1024, 1000, 256, 2048])
def test_fastagc_s16_fused_is_bit_exact(gpu, oracle, block):
    rng = np.random.default_rng(block)
    ch, nb = 5, 37
    x = (rng.uniform(-1, 1, (ch, nb * block)) * rng.uniform(0.01, 3.0, (ch, 1))).astype(np.float32)
    x[1, 3 * block:5 * block] = 0.0                                        # silence: gain capped at 50
    cut = 11 * block
    y1, st, hist = gpu.fastagc_bank_f_s16(_dev(x[:, :cut]), block, 0.8)
    y2, _, _ = gpu.fastagc_bank_f_s16(_dev(x[:, cut:]), block, 0.8, state=st, hist=hist)            # streamed in two calls
    got = np.concatenate([y1.cpu().numpy(), y2.cpu().numpy()], axis=1)
    for c in range(ch):
        want = oracle.convert_f_s16(oracle.fastagc_ff(x[c], block, 0.8))
        assert np.array_equal(got[c], want), (block, c)
