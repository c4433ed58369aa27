"""CPU stepping of the CUDA kernels' __host__ __device__ cores (tests/emu) against the oracle.

Not a product path: tests/emu/libemu.so is a test harness built from the same headers the kernels
use.  It proves index math and arithmetic before GPU time is spent; the real parity tests are the
`-m gpu` ones, which call the kernels through the C ABI."""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import assert_frames_equal
from quant_rule import check_q8
from snout_b200 import chanplan, synth

P = lambda a: a.ctypes.data_as(ctypes.c_void_p)


def _whiten_words(oracle_mod):
    wh, crc, ci = oracle_mod.ble_tables("port")
    w = np.zeros((40, 44), dtype=np.uint8)
    w[:, :42] = wh
    return w.view("<u4").reshape(40, 11).copy(), crc, ci


def _back(emu, oracle_mod, bits, wpp, n_out, ch, m_origin=0, n_windows=None, first_window=0):
    wh11, crc, ci = _whiten_words(oracle_mod)
    if n_windows is None:
        n_windows = (n_out - m_origin + 8191) // 8192
    out = np.zeros(8192, dtype=oracle_mod.FRAME_DTYPE)
    nc = ctypes.c_int(0)
    n = emu.emu_ble_back(P(bits), ctypes.c_uint32(wpp), n_out, m_origin, n_windows, ctypes.c_uint32(first_window), ch,
                         ctypes.c_uint32(0x8E89BED6), ctypes.c_uint32(0xFFFFFFFF), ctypes.c_uint32(ci), P(crc), P(wh11),
                         P(out), 8192, ctypes.byref(nc))
    return out[:n].copy()


def _slice_nb(emu, q_or_x, scale):
    x = np.ascontiguousarray(q_or_x, dtype=np.float32).reshape(-1)
    n = len(x) // 2
    wpp = emu.emu_bits_words_for(n)
    bits = np.zeros(wpp, dtype=np.uint32)
    q8 = np.zeros((n, 2), dtype=np.int8)
    emu.emu_ble_slice_nb(P(x), ctypes.c_int64(n), ctypes.c_float(scale), P(bits), ctypes.c_uint32(wpp), P(q8))
    return bits, wpp, q8


def test_fft_codelets(emu):
    rng = np.random.default_rng(0)
    for n, fn in ((48, emu.emu_idft48), (96, emu.emu_idft96)):
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        y = np.zeros(n, dtype=np.complex64)
        fn(P(x), P(y))
        ref = np.fft.ifft(x.astype(np.complex128)) * n
        assert np.abs(y - ref).max() / np.abs(ref).max() < 1e-6


def test_bin_to_channel_map(emu):
    seen = {}
    for q in range(48):
        ch = emu.emu_ble_channel_of_q(q)
        if ch >= 0:
            assert chanplan.ble_channel_bin(ch) == 2 * q
            seen[ch] = q
    assert sorted(seen) == list(range(40))


def test_nb_slicer_and_back_end_golden(emu, oracle_mod, golden):
    g = golden("btle_sample_iq_4msps.npz")
    bits, wpp, q8 = _slice_nb(emu, g["iq"].astype(np.float32) / 128.0, 128.0)
    assert np.array_equal(q8, g["iq"])
    assert_frames_equal(_back(emu, oracle_mod, bits, wpp, len(q8), 37), g["frames"], what="golden capture")


def test_back_end_window_boundary(emu, oracle_mod, golden):
    g = golden("btle_sample_iq_4msps.npz")["iq"]
    b = golden("btle_boundary_ref.npz")
    for d in range(403, 414):
        gd = np.concatenate([np.zeros((d, 2), np.int8), g[:200_000]])
        bits, wpp, _ = _slice_nb(emu, gd.astype(np.float32) / 128.0, 128.0)
        assert_frames_equal(_back(emu, oracle_mod, bits, wpp, len(gd), 37), b[f"frames_{d}"], what=f"delay {d}")


@pytest.mark.parametrize("seed,ch,esn0", [(1001, 37, 30.0), (1002, 38, 24.0), (1004, 5, 26.0)])
def test_back_end_synthetic(emu, oracle_mod, golden, seed, ch, esn0):
    cap = synth.ble_capture(n=600_000, channel=ch, seed=seed, esn0_db=esn0)
    bits, wpp, q8 = _slice_nb(emu, np.ascontiguousarray(cap.iq).view(np.float32), 128.0)
    assert np.array_equal(q8, oracle_mod.ble_quantize(cap.iq, 128.0))
    assert_frames_equal(_back(emu, oracle_mod, bits, wpp, len(q8), ch), golden("btle_synth_ref.npz")[f"frames_{seed}"],
                        what=f"seed {seed}")


def test_back_end_shard_origin(emu, oracle_mod):
    """A shard that starts 128 samples before window 3 must report exactly the frames of windows 3..5."""
    cap = synth.ble_capture(n=8192 * 8, channel=37, seed=9, esn0_db=30, gap=(100, 1500))
    q = oracle_mod.ble_quantize(cap.iq, 128.0)
    want = oracle_mod.ble_decode(q, 37, first_window=3, n_windows=3)
    lo = 3 * 8192 - 128
    part = q[lo:]
    bits, wpp, _ = _slice_nb(emu, part.astype(np.float32) / 128.0, 128.0)
    got = _back(emu, oracle_mod, bits, wpp, len(part), 37, m_origin=128, n_windows=3, first_window=3)
    assert len(want) > 3
    assert_frames_equal(got, want, what="shard")


@pytest.mark.parametrize("nt,name", [(16, "BLE_384"), (32, "BLE_768")])
def test_pfb_tile_kernel(emu, oracle_mod, nt, name):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from gen_tables import PFB_DESIGNS, kaiser_lowpass
    h = kaiser_lowpass(*PFB_DESIGNS[name])
    hf = h.astype(np.float32)
    rho = np.array([hf[r + 24 * d] for r in range(24) for d in range(nt)], dtype=np.float32)
    cap = synth.wideband_capture(seconds=0.0025, kind="ble", seed=4000, gap=(200, 2000))
    x = np.ascontiguousarray(cap.iq)[: 24 * 8192 - 24 * 40]          # ragged: n_out = 8152, last tile partial
    n_in = len(x)
    n_out = n_in // 24
    T, stride = 32, emu.emu_pfb_ble_stride()
    assert stride == 31
    tiles = (n_out + stride - 1) // stride
    wpp, lead = emu.emu_bits_words_for(n_out), emu.emu_bits_lead_words()
    bits = np.zeros((40, wpp), dtype=np.uint64)                      # 64-bit scratch so that shifted words can spill
    q8 = np.zeros((40, tiles * stride + 1, 2), dtype=np.int8)
    raw = np.zeros((40, tiles * stride + 1), dtype=np.complex64)
    xf = x.view(np.float32)
    for t in range(tiles):
        w = np.zeros(40, dtype=np.uint32)
        q = np.zeros((40, T, 2), dtype=np.int8)
        r = np.zeros((40, T), dtype=np.complex64)
        emu.emu_pfb_ble_tile(nt, P(xf), ctypes.c_int64(n_in), n_out, t, P(rho), ctypes.c_float(100.0), P(w), P(q), P(r))
        g0 = t * stride
        wi, off = lead + (g0 >> 5), g0 & 31                          # what the kernel's two atomicOr do
        sh = w.astype(np.uint64) << np.uint64(off)
        bits[:, wi] |= sh & np.uint64(0xFFFFFFFF)
        bits[:, wi + 1] |= sh >> np.uint64(32)
        if t:                                                        # last sample of a tile == sample 0 of the next
            assert np.array_equal(q8[:, g0], q[:, 0])
        q8[:, g0:g0 + T] = q
        raw[:, g0:g0 + T] = r
    bits = bits.astype(np.uint32)
    assert not q8[:, n_out:].any()                                   # beyond the capture: zeros
    q8, raw = q8[:, :n_out], raw[:, :n_out]
    yd = oracle_mod.pfb(x, h, [chanplan.ble_channel_bin(c) for c in range(40)])
    rms = np.sqrt(np.mean(np.abs(yd) ** 2))
    assert np.abs(raw - yd).max() / rms < 1e-4                       # stated channelizer tolerance
    check_q8(q8, raw, yd, 100.0, what=f"{name} tile harness")
    n_frames = 0
    for c in range(40):
        b2, _, _ = _slice_nb(emu, q8[c].astype(np.float32) / 128.0, 128.0)
        assert np.array_equal(b2, bits[c]), f"slicer words of channel {c}"
        got = _back(emu, oracle_mod, np.ascontiguousarray(bits[c]), wpp, n_out, c)
        assert_frames_equal(got, oracle_mod.ble_decode(q8[c], c), what=f"channel {c}")
        n_frames += len(got)
    assert n_frames > 100


def test_zigbee_cores(emu, oracle_mod):
    cap = synth.zigbee_capture(n=400_000, channel=11, seed=2001, esn0_db=15.0)
    x = np.ascontiguousarray(cap.iq).view(np.float32)
    n = len(cap.iq)
    f = np.zeros(n, dtype=np.float32)
    z = np.zeros(n, dtype=np.float32)
    emu.emu_zb_quad(P(x), ctypes.c_int64(n), P(f))
    assert np.array_equal(f, oracle_mod.zb_quad_demod(cap.iq))       # bit exact
    emu.emu_zb_dc(P(f), ctypes.c_int64(n), P(z))
    assert np.array_equal(z, oracle_mod.zb_dc_remove(f))
    out = np.zeros(1024, dtype=oracle_mod.FRAME_DTYPE)
    for seg, pre in ((65536, 4096), (4096, 2048), (8192, 2048)):
        nseg = -(-n // seg)
        nch = np.zeros(nseg, dtype=np.int64)
        k = emu.emu_zb_chains(P(z), n, 0, n, seg, pre, ctypes.c_uint32(0), 10, 11, P(out), 1024, P(nch))
        want = oracle_mod.zb_receive(cap.iq, 11, segment=seg, prehalo=pre)
        assert len(want) > 5
        assert_frames_equal(out[:k], want, what=f"zigbee chains {seg}/{pre}")
        # every chain stops at the very chip the oracle's chip-by-chip sink stops at
        for c in range(nseg):
            lo, hi = c * seg, min(n, (c + 1) * seg)
            _, ck, _ = oracle_mod.zb_chain(z, max(0, lo - pre), min(n, hi + 16448), lo, hi, want_chips=True, hold=lo - 1024)
            assert nch[c] == len(ck), (seg, c, nch[c], len(ck))


@pytest.mark.parametrize("nt,name", [(16, "ZB_384"), (32, "ZB_768")])
def test_pfb_zb_tile_kernel(emu, oracle_mod, nt, name):
    """Wideband Zigbee front end: channel streams within tolerance of the CPU channelizer statement;
    discriminator bit-identical to the oracle's quadrature demod of the kernel's own (rotated) streams."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from gen_tables import PFB_DESIGNS, kaiser_lowpass
    h = kaiser_lowpass(*PFB_DESIGNS[name])
    hf = h.astype(np.float32)
    rho = np.array([hf[r + 24 * d] for r in range(24) for d in range(nt)], dtype=np.float32)
    cap = synth.wideband_capture(seconds=0.0041, kind="zigbee", seed=3000, esn0_db=20.0, gap=(300, 2500))
    x = np.ascontiguousarray(cap.iq)[: 24 * 16000]
    n_in, n_out = len(x), len(x) // 24
    stride = emu.emu_pfb_tile_stride()
    tiles = max(1, (n_out - 1 + stride - 1) // stride)
    f = np.zeros((16, tiles * stride + 1), dtype=np.float32)
    y = np.zeros((16, tiles * stride + 1), dtype=np.complex64)
    xf = x.view(np.float32)
    for t in range(tiles):
        fo = np.zeros((16, stride), dtype=np.float32)
        yo = np.zeros((16, 128), dtype=np.complex64)
        emu.emu_pfb_zb_tile(nt, P(xf), ctypes.c_int64(n_in), n_out, t, P(rho), P(fo), P(yo))
        f[:, t * stride + 1:(t + 1) * stride + 1] = fo
        y[:, t * stride:t * stride + 128] = yo
    f, y = f[:, :n_out], y[:, :n_out]
    bins = [emu.emu_zb_bin_of_slot(c) for c in range(16)]
    assert bins == [chanplan.zigbee_channel_bin(11 + c) for c in range(16)]
    yd = oracle_mod.pfb(x, h, bins)
    assert np.abs(y - yd).max() / np.sqrt(np.mean(np.abs(yd) ** 2)) < 1e-4
    ok = tot = 0
    for c in range(16):
        assert np.array_equal(f[c], oracle_mod.zb_quad_demod(y[c])), f"discriminator of slot {c}"
        fr = oracle_mod.zb_receive_z(oracle_mod.zb_dc_remove(f[c]), 11 + c)
        truth = {bytes(t.data) for t in cap.truth if t.channel == 11 + c and t.start + 4300 < n_out}
        ok += len(truth & {bytes(q["bytes"][:q["len"]]) for q in fr if q["crc_ok"]})
        tot += len(truth)
    assert tot >= 8 and ok >= 0.9 * tot, (ok, tot)


def test_zb_chain_order_key(emu, oracle_mod):
    """k_zb_order's key (csrc/zb.cuh zb_chain_key): which chains k_zb_rx hands out first.  It is a scheduling hint -- no record
    depends on it (GPU test test_zb_chain_order_is_a_scheduling_hint_only) -- but it indexes the counting sort, so its range and
    its meaning are pinned here: 0 when the air is idle at the end of the chain's body or has been busy without a break since
    two blocks before the body, else the number of consecutive busy block ends from the end of the body on (at most 9)."""
    import ctypes
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    K = emu.emu_zb_keys()
    assert K == 10

    def key(busy, origin, body, segment, seg):
        return emu.emu_zb_chain_key(P(busy), len(busy), origin, body, segment, seg)

    def want(busy, origin, body, segment, seg):
        lo = origin + seg * segment
        hi = min(lo + segment, origin + body)
        if hi <= lo or hi % 2048 or lo % 2048:
            return 0
        kb, kl = hi // 2048 - 1, lo // 2048 - 1
        if kb < 0 or kb >= len(busy) or not busy[kb]:
            return 0
        if kl >= 1 and all(busy[j] for j in range(kl - 1, kb)):
            return 0
        k, j = 0, kb
        while j < len(busy) and busy[j] and k < K - 1:
            k, j = k + 1, j + 1
        return k

    rng = np.random.default_rng(11)
    for trial in range(300):
        nb = int(rng.integers(4, 80))
        busy = (rng.random(nb) < rng.choice([0.1, 0.5, 0.9])).astype(np.uint8)
        segment = int(rng.choice([2048, 4096, 8192, 16384]))
        origin = int(rng.choice([0, 2048 * 3, 2048 * 49]))
        body = nb * 2048 - origin - int(rng.choice([0, 0, 700]))
        if body <= 0:
            continue
        for seg in range(-(-body // segment)):
            k = key(busy, origin, body, segment, seg)
            assert 0 <= k < K and k == want(busy, origin, body, segment, seg), (trial, seg, k)
    # a frame that starts inside the body and runs on for three blocks past it; the same frame seen by the NEXT chain (on the air
    # since before its body) is not that chain's to decode
    busy = np.zeros(20, np.uint8); busy[5:9] = 1            # busy at the ends of blocks 5..8 = samples 12288 .. 18432
    assert key(busy, 0, 20 * 2048, 4096, 2) == 4            # body [8192, 12288): ends busy, then 3 more busy block ends
    assert key(busy, 0, 20 * 2048, 4096, 3) == 2            # body [12288, 16384): idle at 10240, so it may be this chain's: 2 more
    busy[3:9] = 1                                           # ... on the air since 8192: not the chain's to decode
    assert key(busy, 0, 20 * 2048, 4096, 3) == 0
    # the discriminator statistics the busy flag rests on: O-QPSK moves by +-pi/4 per sample, noise is uniform in (-pi, pi)
    msk = np.full(64, np.pi / 4, np.float32) * rng.choice([-1.0, 1.0], 64).astype(np.float32)
    noise = rng.uniform(-np.pi, np.pi, 64).astype(np.float32)
    gfsk = np.full(64, 0.39, np.float32)
    assert emu.emu_zb_block_busy(P(msk)) == 1 and emu.emu_zb_block_busy(P(noise)) == 0 and emu.emu_zb_block_busy(P(gfsk)) == 0
    assert emu.emu_zb_block_busy(P(np.zeros(64, np.float32))) == 0


def test_transpose_step_rotate_select_identity():
    """csrc/pfb.cuh transpose_step on the device is one rotate + one bitwise select; on the host (and in the harness) it is the
    two-sided shift form it replaced.  They are the same function: under m no bit of y >> j wraps, under ~m none of y << j does."""
    rng = np.random.default_rng(5)
    ror = lambda v, r: ((v >> np.uint32(r)) | (v << np.uint32(32 - r))) & np.uint32(0xFFFFFFFF) if r % 32 else v   # noqa: E731
    for j, m in ((8, 0x00FF00FF), (4, 0x0F0F0F0F), (2, 0x33333333), (1, 0x55555555), (16, 0x0000FFFF)):
        m = np.uint32(m)
        x = rng.integers(0, 1 << 32, 2000, dtype=np.uint64).astype(np.uint32)
        y = rng.integers(0, 1 << 32, 2000, dtype=np.uint64).astype(np.uint32)
        for hi in (False, True):
            two_sided = ((x & ~m) | ((y >> np.uint32(j)) & m)) if hi else ((x & m) | ((y << np.uint32(j)) & ~m))
            keep = ~m if hi else m
            rot = ror(y, j if hi else 32 - j)
            assert np.array_equal(two_sided, (x & keep) | (rot & ~keep)), (j, hi)
