"""The BLE back end (k_aa_search, k_aa_fill, k_ble_decode, k_ble_resolve, snrx_ble_follow) driven with constructed bit streams.

tests/ble_bits.py builds int8 captures whose slicer decisions are exactly a chosen bit stream, so the order-dependent rules
of receiver() can be put to work where natural captures rarely take them: virtual matches at search origins, resumes after
a gated header, the last start positions of a window (no frame can reach the demodulation limit), window edges at every phase, captures cut inside a frame, address look-alikes
inside frames, and the candidate and frame capacities.  Every result is compared with ble_expected (the restatement
oracle/ble_oracle.c, and the unmodified btle_rx.c wherever it was compiled).

The unmarked tests step the kernels' own cores on the CPU (tests/emu); the gpu tests run the same streams through the engine."""
import ctypes

import numpy as np
import pytest

import ble_bits as bb
from conftest import assert_frames_equal, ble_expected

P = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
W = bb.WINDOW


# ------------------------------------------------------------------------------------------------ the stream families
def _dense():
    return [bb.dense(s) for s in range(260)]


def _near():
    return [bb.near_misses(s) for s in range(90)]


def _lookalike():
    return [bb.lookalikes(s) for s in range(80)]


def _edges():
    return [bb.window_edges(1000 * k + o, W * k - 160 + o) for k in (0, 1, 2) for o in range(169)]


def _ends():
    out = [bb.capture_end(100 * c + s, c) for c in range(1, 47) for s in range(2)]
    out += [bb.short(5000 + r, 3 * W + 400 + r) for r in range(128)]            # every residue mod 4, 32 and 128
    out += [bb.short(6000 + n, n) for n in (1, 2, 3, 5, 31, 33, 127, 129, 500, 1471, 1473, 4096, W - 1, W, W + 1)]
    return out


def _virtual():
    return [bb.virtual_history(31 * z + s, z) for z in range(32) for s in range(6)]


def _patho():
    return [bb.pathological(s, k) for k in ("zeros", "ones", "x55", "xaa", "survivors") for s in range(4)]


FAMILIES = {"dense": _dense, "near_misses": _near, "lookalikes": _lookalike, "window_edges": _edges,
            "capture_end": _ends, "virtual_history": _virtual, "pathological": _patho}
# frames each family must reach: the CPU part compares at least 10^4 frames in all
FAMILY_MIN = {"dense": 4500, "near_misses": 1300, "lookalikes": 1300, "window_edges": 5500, "capture_end": 4000,
              "virtual_history": 3000, "pathological": 150}
assert sum(FAMILY_MIN.values()) >= 10_000


def _want(oracle_mod, iq, par, **kw):
    return ble_expected(oracle_mod, iq, par["channel"], aa=par["aa"], crc_init=par["crc_cmdline"], aa_mask=par["aa_mask"], **kw)


# ------------------------------------------------------------------------------------------------ CPU: the kernels' cores
@pytest.fixture(scope="module")
def tabs(oracle_mod):
    wh, crc, _ = oracle_mod.ble_tables("port")
    w = np.zeros((40, 44), dtype=np.uint8)
    w[:, :42] = wh
    return w.view("<u4").reshape(40, 11).copy(), crc, oracle_mod.FRAME_DTYPE


def _emu_back(emu, tabs, x, par, m_origin=0, n_windows=None, first_window=0, cap=1 << 16, out=None):
    """emu_ble_slice_nb on cf32 q / 128, then emu_ble_back; returns (frames, bits, number of frames found)."""
    wh11, crc, dtype = tabs
    n = len(x)
    xf = np.ascontiguousarray(x, dtype=np.float32).reshape(-1) / np.float32(128.0)
    wpp = emu.emu_bits_words_for(n)
    bits = np.zeros(wpp, dtype=np.uint32)
    emu.emu_ble_slice_nb(P(xf), ctypes.c_int64(n), ctypes.c_float(128.0), P(bits), ctypes.c_uint32(wpp), None)
    if n_windows is None:
        n_windows = (n - m_origin + W - 1) // W
    if out is None:
        out = np.zeros(cap, dtype=dtype)
    k = emu.emu_ble_back(P(bits), ctypes.c_uint32(wpp), n, m_origin, n_windows, ctypes.c_uint32(first_window), par["channel"],
                         ctypes.c_uint32(par["aa"]), ctypes.c_uint32(par["aa_mask"]),
                         ctypes.c_uint32(bb.crc_internal(par["crc_init"])), P(crc), P(wh11), P(out), cap, None)
    return out[:min(k, cap)].copy(), bits, k


def test_construction_is_exact():
    """Every cross product of a constructed capture is +-4096 with the sign of b; packing follows BitsLayout."""
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 31, 32, 33, 1000):
        b = rng.integers(0, 2, n, dtype=np.uint8)
        bb.check_iq(b, bb.bits_to_iq(b))
    b = np.zeros(70, np.uint8)
    b[[0, 31, 32, 69]] = 1
    w = bb.pack_words(b, 4, 4 + 3 + 64)
    assert w[:4].tolist() == [0, 0, 0, 0] and w[4] == 0x80000001 and w[5] == 1 and w[6] == 1 << 5 and not w[7:].any()
    # the frame is the address LSB first, then whiten(header | payload | crc24) LSB first
    f = bb.frame_symbols(37, b"\x02\x00", b"", aa=0x8E89BED6)
    assert f[:32].tolist() == [(0x8E89BED6 >> k) & 1 for k in range(32)] and len(f) == 32 + 8 * 5


@pytest.mark.parametrize("family", list(FAMILIES))
def test_family_cpu(emu, oracle_mod, tabs, family):
    total = 0
    for iq, par in FAMILIES[family]():
        bb.check_iq(par["bits"], iq)
        got, bits, _ = _emu_back(emu, tabs, iq, par)
        assert np.array_equal(bits, bb.pack_words(par["bits"], 4, len(bits))), "harness slicer words"
        what = f"{family}: n = {len(iq)}, channel {par['channel']}, aa {par['aa']:#010x}, mask {par['aa_mask']:#010x}"
        assert_frames_equal(got, _want(oracle_mod, iq, par), what=what)
        total += len(got)
    print(f"{family}: {total} frames compared")
    assert total >= FAMILY_MIN[family], (family, total)


def test_shards_cpu(emu, oracle_mod, tabs):
    """Shards (m_origin, first_window, n_windows) against the oracle's windows of the whole capture."""
    total = 0
    for seed in range(30):
        iq, par = bb.dense(700 + seed, n=int(np.random.default_rng(seed).integers(3 * W, 6 * W)))
        nw = (len(iq) + W - 1) // W
        rng = np.random.default_rng(seed)
        cuts = sorted(set([0, nw] + rng.integers(1, nw, 2).tolist()))
        parts = []
        for w0, w1 in zip(cuts[:-1], cuts[1:]):
            lo = max(0, w0 * W - 128)
            hi = min(len(iq), w1 * W + 2048)
            got, _, _ = _emu_back(emu, tabs, iq[lo:hi], par, m_origin=w0 * W - lo, n_windows=w1 - w0, first_window=w0)
            want = oracle_mod.ble_decode(iq, par["channel"], aa=par["aa"], crc_init=par["crc_cmdline"], aa_mask=par["aa_mask"],
                                         first_window=w0, n_windows=w1 - w0)
            assert_frames_equal(got, want, what=f"seed {seed}, windows {w0}..{w1}")
            parts.append(got)
        assert_frames_equal(np.concatenate(parts), _want(oracle_mod, iq, par), what=f"seed {seed}: shards vs whole")
        total += sum(len(p) for p in parts)
    assert total > 800


@pytest.mark.parametrize("channel,length", [(37, 37), (12, 31)])
def test_farthest_frame_of_a_window(emu, oracle_mod, tabs, channel, length):
    """The search of a window reports access-address bit 0 at most 8191 samples past the window start (t < slots), so a frame
    reaches at most 2 * 8191 + 384 + 64 * (length + 3) = 19326 int8 into the window: below the demodulation limit (19392), which
    therefore never cuts a frame.  The longest frames at the last start positions of windows 0..2 are reported whole in their
    window (and found again by the next window, from its zeroed history, when z allows)."""
    for k in range(3):
        for off in range(8184, 8192):
            rng = np.random.default_rng(off + 10 * k)
            par = dict(channel=channel, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
            b = rng.integers(0, 2, W * (k + 2), dtype=np.uint8)
            bb.plant(b, W * k + off, bb.random_frame(rng, channel, bb.ADV_AA, 0x555555, length=length, crc_ok=True))
            iq, par = bb._finish(b, par)
            want = _want(oracle_mod, iq, par)
            got, _, _ = _emu_back(emu, tabs, iq, par)
            assert_frames_equal(got, want, what=f"window {k}, offset {off}")
            mine = want[(want["sample_index"] == W * k + off) & (want["window"] == k)]
            assert len(mine) == 1 and mine[0]["crc_ok"] == 1 and mine[0]["len"] == length + 5


def test_frame_capacity_guard_cpu(emu, oracle_mod, tabs):
    """With room for fewer frames than it finds, the back end counts them all and writes none past its capacity."""
    iq, par = bb.dense(3, n=30_000)
    full, _, n = _emu_back(emu, tabs, iq, par)
    assert n == len(full) > 20
    out = np.zeros(n, dtype=tabs[2])
    out[n - 1]["sample_index"] = -12345
    out[n - 1]["bytes"][:] = 0xA5
    canary = out[n - 1].copy()
    got, _, k = _emu_back(emu, tabs, iq, par, cap=n - 1, out=out)
    assert k == n and out[n - 1] == canary
    assert_frames_equal(got, full[:n - 1], what="capped")


def test_capacity_stream_counts():
    """The capacity streams hold exactly the number of candidates they are built with (counted here independently)."""
    for k in (24, 31, 1000):
        b = bb.capacity_stream(k, seed=k)
        assert bb.count_candidates(b, bb.ADV_AA, bb.mask_hi(bb.ADV_AA, 0xFFFFFFFF)) == k


@pytest.mark.parametrize("aa,mask", [(0x50000000, 0x0000FFFF), (0x50000000, 0xAF258C8F), (0, 0xFFFFFFFF)])
def test_address_without_a_compared_one_bit(emu, oracle_mod, tabs, aa, mask):
    """aa & mask == 0 (the engine refuses it, DESIGN §4): the reference, fed zero samples past the capture as its harness
    does, then reports frames that start past the end of the capture, where the sliding correlation has no start positions,
    so the kernels cannot agree.  Inside the capture they do."""
    n_past = 0
    for seed in (17, 47, 57, 77):
        iq, par = bb.dense(seed, n=30_000 + 1000 * (seed % 6), aa=aa, aa_mask=mask)
        want = _want(oracle_mod, iq, par)
        got, _, _ = _emu_back(emu, tabs, iq, par)
        past = want["sample_index"] >= len(iq)
        n_past += int(past.sum())
        assert_frames_equal(got, want[~past], what=f"seed {seed}: inside the capture")
    assert n_past > 0


# ------------------------------------------------------------------------------------------------ GPU: the engine
@pytest.fixture(scope="module")
def Engine():
    from snout_b200 import _abi
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"

    def make(par, **kw):
        kw.setdefault("max_frames", 1 << 13)
        return RxEngine("ble_nb", channel=par["channel"], access_addr=par["aa"], crc_init=par["crc_cmdline"],
                        access_mask=par["aa_mask"], **kw)
    return make


def _gpu_streams():
    """A slice of every family: what runs through the engine one capture at a time."""
    out = []
    out += [bb.dense(s) for s in range(0, 260, 26)]
    out += [bb.near_misses(s) for s in (1, 2)] + [bb.lookalikes(s) for s in (1, 2)]
    out += [bb.window_edges(1000 * k + o, W * k - 160 + o) for k, o in ((0, 0), (1, 37), (1, 160), (2, 168), (2, 90))]
    out += [bb.capture_end(100 * c, c) for c in (1, 13, 46)] + [bb.short(6000 + n, n) for n in (1, 33, 1473, W + 1)]
    out += [bb.virtual_history(31 * z, z) for z in (0, 1, 7, 16, 30, 31)]
    out += [bb.pathological(0, k) for k in ("ones", "x55", "survivors")]
    return out


@pytest.mark.gpu
def test_families_gpu(Engine, oracle_mod):
    from snout_b200 import _abi
    total = 0
    for i, (iq, par) in enumerate(_gpu_streams()):
        want = _want(oracle_mod, iq, par)
        what = f"stream {i}: n = {len(iq)}, channel {par['channel']}, aa {par['aa']:#010x}, mask {par['aa_mask']:#010x}"
        with Engine(par, max_samples=len(iq)) as e:
            assert_frames_equal(e.run(iq), want, what=what + " sc8")
            assert_frames_equal(e.run(iq.astype(np.float32).view(np.complex64)[:, 0] / np.float32(128.0)), want, what=what + " cf32")
        with Engine(par, max_samples=len(iq), keep_streams=True) as e:
            assert_frames_equal(e.run(iq), want, what=what + " keep_streams")
            bits = e.debug_stage(_abi.STAGE_BLE_BITS)[0, 0]
        assert np.array_equal(bits, bb.pack_words(par["bits"], 4, 4 + (len(iq) + 31) // 32 + 64)), what + ": bit stream"
        total += len(want)
    print(f"{total} frames compared")
    assert total > 400


def _batch_par():
    return dict(channel=5, aa=0x71764129, aa_mask=0xFFFFFFFF, crc_init=0x123456, crc_cmdline=bb.crc_cmdline(0x123456))


def _batch_streams(par, n_caps=64):
    fixed = {k: par[k] for k in ("channel", "aa", "aa_mask", "crc_init")}
    makers = [lambda s: bb.dense(s, **fixed), lambda s: bb.near_misses(s, **fixed), lambda s: bb.lookalikes(s, **fixed),
              lambda s: bb.window_edges(s, W * (s % 3) - 160 + (s * 7) % 169, **fixed),
              lambda s: bb.capture_end(s, 1 + s % 46, **fixed), lambda s: bb.short(s, 1 + (s * 997) % (2 * W), **fixed),
              lambda s: bb.pathological(s, "survivors", **fixed)]
    return [makers[i % len(makers)](900 + i) for i in range(n_caps)]


@pytest.mark.gpu
def test_batch_of_64_gpu(Engine, oracle_mod):
    """64 captures of different families and ragged lengths (zero-filled to the batch length) in one batch, with non-zero
    stride padding: per capture, the records of a single-capture run and the oracle's, with the right capture_id."""
    par = _batch_par()
    streams = _batch_streams(par)
    n = max(len(iq) for iq, _ in streams)
    stride = n + 38
    x = np.random.default_rng(5).integers(-128, 128, (64, stride, 2)).astype(np.int8)
    for k, (iq, _) in enumerate(streams):
        x[k, :n] = 0
        x[k, :len(iq)] = iq
    with Engine(par, max_samples=n, max_captures=64, max_frames=1 << 15) as e:
        got = e.run(x, n_samples=n, stride=stride)
        total = 0
        for k, (iq, p) in enumerate(streams):
            mine = got[got["capture_id"] == k]
            want = _want(oracle_mod, iq, p)
            assert_frames_equal(mine, want, what=f"capture {k} of the batch")
            assert_frames_equal(e.run(iq), want, what=f"capture {k} alone")
            total += len(want)
        assert np.all(np.diff(got["capture_id"].astype(np.int64)) >= 0)
    assert total > 500


@pytest.mark.gpu
def test_follow_gpu(Engine, oracle_mod):
    """follow(aa, crc_init) for 32 addresses planted in the same batch, aa with 0..31 trailing zeros (z = 0..31)."""
    rng = np.random.default_rng(77)
    pairs = []
    for z in range(32):
        aa, _ = bb.virtual_aa(rng, z)
        pairs.append((aa, int(rng.integers(0, 1 << 24))))
    caps = []
    for c in range(3):
        n = 3 * W + 1000 * c
        b = rng.integers(0, 2, n, dtype=np.uint8)
        s = int(rng.integers(-100, 50))
        while s < n:
            aa, ci = pairs[int(rng.integers(0, 32))]
            bb.plant(b, s, bb.random_frame(rng, 17, aa, ci))
            s += int(rng.integers(40, 400))
        caps.append(bb.effective_bits(b))
    n = max(len(b) for b in caps)
    x = np.zeros((3, n, 2), np.int8)
    iqs = []
    for c, b in enumerate(caps):
        iq = bb.bits_to_iq(b)
        x[c, :len(iq)] = iq
        iqs.append(x[c])
    par = dict(channel=17, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555, crc_cmdline=0x555555)
    total = 0
    with Engine(par, max_samples=n, max_captures=3) as e:
        e.run(x)
        for aa, ci in pairs:
            got = e.follow(aa, bb.crc_cmdline(ci))
            want = []
            for c in range(3):
                w = oracle_mod.ble_decode(iqs[c], 17, aa=aa, crc_init=bb.crc_cmdline(ci))
                w["capture_id"] = c
                want.append(w)
            want = np.concatenate(want)
            assert_frames_equal(got, want, what=f"follow {aa:#010x}")
            assert np.array_equal(got["capture_id"], want["capture_id"])
            total += len(want)
    assert total > 300


@pytest.mark.gpu
def test_shards_gpu(Engine, oracle_mod):
    """A dense stream cut at window boundaries (128-sample pre halo, 2048-sample post halo) equals the whole capture."""
    iq, par = bb.dense(4242, n=7 * W + 555)
    want = _want(oracle_mod, iq, par)
    with Engine(par, max_samples=len(iq)) as e:
        whole = e.run(iq)
        parts = []
        for w0, w1 in ((0, 2), (2, 3), (3, 6), (6, 8)):
            lo, hi = max(0, w0 * W - 128), min(len(iq), w1 * W + 2048)
            body = min((w1 - w0) * W, len(iq) - w0 * W)
            parts.append(e.run(iq[lo:hi].copy(), shard=dict(pre_samples=w0 * W - lo, body_samples=body, first_window=w0)))
    assert_frames_equal(whole, want, what="whole vs oracle")
    assert_frames_equal(np.concatenate(parts), whole, what="shards vs whole")
    assert len(want) > 40


@pytest.mark.gpu
def test_candidate_capacity_gpu(Engine, oracle_mod):
    """max_frames = 2^14 gives a candidate capacity of 2^16: exactly 2^16 candidates decode like the oracle; one more fails
    the poll with SNRX_EOVERFLOW; the next ordinary batch on the same engine is right again."""
    from snout_b200._abi import SnrxError
    cap = 1 << 16
    par = dict(channel=37, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555, crc_cmdline=0x555555)
    full = bb.capacity_stream(cap, seed=1)
    over = bb.capacity_stream(cap + 1, seed=2)
    mh = bb.mask_hi(bb.ADV_AA, 0xFFFFFFFF)
    assert bb.count_candidates(full, bb.ADV_AA, mh) == cap and bb.count_candidates(over, bb.ADV_AA, mh) == cap + 1
    iq_full, iq_over = bb.bits_to_iq(full), bb.bits_to_iq(over)
    want = _want(oracle_mod, iq_full, par)
    assert 10 <= len(want) <= 1 << 14
    plain, ppar = bb.dense(31, channel=37, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
    with Engine(par, max_samples=len(iq_over), max_frames=1 << 14) as e:
        assert_frames_equal(e.run(iq_full), want, what="at the candidate capacity")
        assert e.stats()["candidates"] == cap
        with pytest.raises(SnrxError) as ex:
            e.run(iq_over)
        assert ex.value.code == -6
        assert_frames_equal(e.run(plain), _want(oracle_mod, plain, ppar), what="after the overflow")


@pytest.mark.gpu
def test_frame_capacity_gpu(Engine, oracle_mod):
    """max_frames equal to the frame count: the frames; one less: SNRX_EOVERFLOW, for poll and for follow."""
    from snout_b200._abi import SnrxError
    iq, par = bb.dense(12, n=40_000, channel=38, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
    want = _want(oracle_mod, iq, par)
    nf = len(want)
    assert nf > 10
    with Engine(par, max_samples=len(iq), max_frames=nf) as e:
        assert_frames_equal(e.run(iq), want, what="max_frames = frames")
    with Engine(par, max_samples=len(iq), max_frames=nf - 1) as e:
        with pytest.raises(SnrxError) as ex:
            e.run(iq)
        assert ex.value.code == -6
    # follow: a batch without a frame of the engine's own address, searched again with the planted one
    fpar = dict(par, aa=0x6B2D94C3)
    iq2, p2 = bb.dense(13, n=40_000, channel=38, aa=fpar["aa"], aa_mask=0xFFFFFFFF, crc_init=0x555555)
    fw = _want(oracle_mod, iq2, p2)
    assert len(oracle_mod.ble_decode(iq2, 38)) == 0 and len(fw) > 10
    for cap, ok in ((len(fw), True), (len(fw) - 1, False)):
        with Engine(par, max_samples=len(iq2), max_frames=cap) as e:
            assert len(e.run(iq2)) == 0
            if ok:
                assert_frames_equal(e.follow(fpar["aa"], 0x555555), fw, what="follow at max_frames")
            else:
                with pytest.raises(SnrxError) as ex:
                    e.follow(fpar["aa"], 0x555555)
                assert ex.value.code == -6


@pytest.mark.gpu
@pytest.mark.parametrize("aa,mask", [(0x50000000, 0x0000FFFF), (0x50000000, 0xAF258C8F), (0x12345678, 0xEDCBA987),
                                     (0, 0xFFFFFFFF)])
def test_address_without_a_compared_one_bit_is_refused(Engine, aa, mask):
    from snout_b200._abi import SnrxError
    par = dict(channel=37, aa=aa, aa_mask=mask, crc_init=0x123456, crc_cmdline=0x123456)
    with pytest.raises(SnrxError) as ex:
        Engine(par, max_samples=1 << 16)
    assert ex.value.code == -1
    iq, p = bb.dense(5, n=20_000, channel=37, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
    with Engine(p, max_samples=len(iq)) as e:
        e.run(iq)
        with pytest.raises(SnrxError) as ex:
            e.follow(0, 0x555555)
        assert ex.value.code == -1
