"""Parity tests proper: the CUDA path, called through the C ABI (snout_b200._abi -> libsnoutrx.so),
against the oracle and the committed reference outputs.  Bit-exact for frames (bytes, channel, CRC
flag, sample index, window, order); stated tolerances for the float stages.

Run on the GPU box with `pytest -m gpu`.  Nothing here reads /root/reference."""
import os

import numpy as np
import pytest

from conftest import assert_frames_equal, ble_expected
from snout_b200 import _abi, chanplan, synth

pytestmark = pytest.mark.gpu

CHAN_TOL = 1e-4          # channelizer: max |err| / rms of the channel streams (BASELINE north_star: rel err <= 1e-4)


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


# ------------------------------------------------------------------------------------ BLE narrow band
def test_ble_nb_golden_capture(Engine, golden):
    g = golden("btle_sample_iq_4msps.npz")
    x = (g["iq"].astype(np.float32) / 128.0).view(np.complex64).reshape(-1)
    with Engine("ble_nb", channel=37, max_samples=len(x), keep_streams=True) as e:
        got = e.run(x)
        assert np.array_equal(e.debug_stage(_abi.STAGE_BLE_Q8)[0, 0], g["iq"])
        st = e.stats()
    assert list(got["sample_index"]) == [97892, 501906, 905891]
    assert_frames_equal(got, g["frames"], what="golden capture vs reference output")
    assert st["frames"] == 3 and st["frames_crc_ok"] == 3 and st["kernel_launches"] >= 6


def test_ble_nb_welcome_vector(Engine, golden):
    g = golden("btle_welcome.npz")
    x = (g["iq"].astype(np.float32) / 256.0).view(np.complex64).reshape(-1)
    with Engine("ble_nb", channel=37, max_samples=4096, quant_scale=256.0) as e:
        assert_frames_equal(e.run(x), g["frames"], what="welcome vector")


@pytest.mark.parametrize("seed", [1001, 1002, 1003, 1004])
def test_ble_nb_synthetic_vs_reference_fixture(Engine, oracle_mod, golden, seed):
    g = golden("btle_synth_ref.npz")
    s, esn0, ch, n = g[f"params_{seed}"]
    cap = synth.ble_capture(n=int(n), channel=int(ch), seed=int(s), esn0_db=float(esn0))
    with Engine("ble_nb", channel=int(ch), max_samples=int(n)) as e:
        got = e.run(cap.iq)
    assert_frames_equal(got, g[f"frames_{seed}"], what=f"seed {seed} vs reference fixture")
    assert_frames_equal(got, ble_expected(oracle_mod, oracle_mod.ble_quantize(cap.iq, 128.0), int(ch)), what="vs oracle")


def test_ble_nb_window_boundary_rule(Engine, golden):
    g = golden("btle_sample_iq_4msps.npz")["iq"]
    b = golden("btle_boundary_ref.npz")
    with Engine("ble_nb", channel=37, max_samples=200_000 + 512) as e:
        for d in range(403, 414):
            gd = np.concatenate([np.zeros((d, 2), np.int8), g[:200_000]])
            if len(gd) % 2:
                gd = np.concatenate([gd, np.zeros((1, 2), np.int8)])
            x = (gd.astype(np.float32) / 128.0).view(np.complex64).reshape(-1)
            assert_frames_equal(e.run(x), b[f"frames_{d}"], what=f"delay {d}")


def test_ble_nb_batch_ragged_and_edge_cases(Engine, oracle_mod):
    n = 8192 * 5 + 1234                      # ragged: not a multiple of the window, nor of 128
    caps = [synth.ble_capture(n=n, channel=12, seed=500 + i, esn0_db=30, gap=(100, 1200)).iq for i in range(5)]
    batch = np.stack(caps)
    with Engine("ble_nb", channel=12, max_samples=n, max_captures=5) as e:
        got = e.run(batch)
        want = []
        for i, c in enumerate(caps):
            f = ble_expected(oracle_mod, oracle_mod.ble_quantize(c, 128.0), 12)
            f["capture_id"] = i
            want.append(f)
        want = np.concatenate(want)
        assert len(want) > 20
        assert_frames_equal(got, want, what="batch of 5 ragged captures")
        assert np.array_equal(got["capture_id"], want["capture_id"])
        # empty / silent / full-scale inputs
        assert len(e.run(np.zeros(n, np.complex64))) == 0
        assert len(e.run(np.zeros(2, np.complex64))) == 0
        rng = np.random.default_rng(7)
        noise = (rng.integers(-128, 128, (n, 2)).astype(np.float32) / 128.0).view(np.complex64).reshape(-1)
        f = e.run(noise)
        assert_frames_equal(f, ble_expected(oracle_mod, oracle_mod.ble_quantize(noise, 128.0), 12), what="noise")
        with pytest.raises(_abi.SnrxError):
            e.run(np.zeros(n + 2, np.complex64))          # over capacity -> SNRX_ERANGE, loudly


def test_ble_nb_sc8_golden_capture(Engine, golden):
    """snrx_process_sc8: the reference's own sample format (int8 I,Q, btle_rx.c:204,489-498) goes in as is."""
    g = golden("btle_sample_iq_4msps.npz")
    with Engine("ble_nb", channel=37, max_samples=len(g["iq"]), keep_streams=True) as e:
        got = e.run(g["iq"])                                     # int8 [n, 2]
        assert np.array_equal(e.debug_stage(_abi.STAGE_BLE_Q8)[0, 0], g["iq"])
        assert e.stats()["kernel_launches"] >= 7                 # + the sc8 expansion kernel
    assert list(got["sample_index"]) == [97892, 501906, 905891]
    assert_frames_equal(got, g["frames"], what="golden capture (sc8) vs reference output")


def test_sc8_equals_cf32_all_paths(Engine):
    """int8 input q and cf32 input q/128 give identical frames: host and device pointers, batches with odd
    lengths and strides, wideband (pipelined staging) and Zigbee."""
    import torch
    rng = np.random.default_rng(3)
    n = 8192 * 6 + 777                       # odd
    caps = [synth.ble_capture(n=n, channel=5, seed=700 + i, esn0_db=30, gap=(100, 1200)).iq for i in range(3)]
    q = np.stack([np.clip(np.rint(c.view(np.float32).reshape(-1, 2) * 128.0), -128, 127).astype(np.int8) for c in caps])
    x = (q.astype(np.float32) / 128.0).view(np.complex64).reshape(3, n)
    qp = np.zeros((3, n + 1, 2), np.int8)     # odd length inside an even stride (captures must stay 16-byte aligned)
    qp[:, :n] = q
    xp = np.zeros((3, n + 1), np.complex64)
    xp[:, :n] = x
    with Engine("ble_nb", channel=5, max_samples=n, max_captures=3) as e:
        want = e.run(xp, n_samples=n, stride=n + 1)
        assert len(want) > 10
        assert_frames_equal(e.run(qp, n_samples=n, stride=n + 1), want, what="sc8 host batch")
        assert_frames_equal(e.run(torch.from_numpy(qp).cuda(), n_samples=n, stride=n + 1), want, what="sc8 device batch")
        with pytest.raises(_abi.SnrxError):
            e.run(q)                                            # odd stride: captures not aligned -> refused loudly
    wb = synth.wideband_capture(seconds=0.02, kind="mixed", seed=5200, esn0_db=25.0, gap=(400, 5000))
    peak = float(np.abs(wb.iq).max())        # an 8-bit wideband digitiser: full scale just above the peak of the sum
    q = np.clip(np.rint(wb.iq.view(np.float32).reshape(-1, 2) * (100.0 / peak)), -128, 127).astype(np.int8)
    x = (q.astype(np.float32) / 128.0).view(np.complex64).reshape(-1)
    for mode in ("ble_wb40", "mixed_wb56"):
        with Engine(mode, max_samples=len(x), zb_segment=16384, quant_scale=128.0 * peak) as e:
            want = e.run(x)
            assert len(want) > 20, mode
            assert_frames_equal(e.run(q), want, what=f"{mode}: sc8 host")
            assert_frames_equal(e.run(torch.from_numpy(q).cuda()), want, what=f"{mode}: sc8 device")
    del rng


def test_ble_nb_device_pointer_equals_host_pointer(Engine):
    import torch
    cap = synth.ble_capture(n=300_000, channel=37, seed=11, esn0_db=30)
    with Engine("ble_nb", channel=37, max_samples=300_000) as e:
        a = e.run(cap.iq)
        t = torch.from_numpy(cap.iq).cuda()
        b = e.run(t)
    assert len(a) > 10
    assert_frames_equal(a, b, what="host vs device input")


def test_ble_nb_shard_equals_whole(Engine, oracle_mod):
    cap = synth.ble_capture(n=8192 * 12, channel=37, seed=9, esn0_db=30, gap=(100, 1500))
    q = oracle_mod.ble_quantize(cap.iq, 128.0)
    with Engine("ble_nb", channel=37, max_samples=8192 * 12) as e:
        whole = e.run(cap.iq)
        parts = []
        for w0, w1 in ((0, 5), (5, 9), (9, 12)):
            lo = max(0, w0 * 8192 - 128)
            hi = min(len(cap.iq), w1 * 8192 + 2048)
            parts.append(e.run(cap.iq[lo:hi].copy(), shard=dict(pre_samples=w0 * 8192 - lo, body_samples=(w1 - w0) * 8192,
                                                               first_window=w0)))
        assert_frames_equal(np.concatenate(parts), whole, what="3 shards vs whole")
    assert_frames_equal(whole, ble_expected(oracle_mod, q, 37), what="whole vs oracle")


def test_ble_nb_full_size_config1(Engine, oracle_mod):
    """BASELINE config 1: 1e7 samples of channel 37.  Full comparison (the oracle takes < 1 s)."""
    cap = synth.ble_capture(n=10_000_000, channel=37, seed=1001, esn0_db=30.0)
    with Engine("ble_nb", channel=37, max_samples=10_000_000) as e:
        got = e.run(cap.iq)
    want = ble_expected(oracle_mod, oracle_mod.ble_quantize(cap.iq, 128.0), 37)
    assert len(want) > 1000
    assert_frames_equal(got, want, what="config 1")
    truth = {bytes(t.data) for t in cap.truth}
    assert len(truth & {bytes(f["bytes"][:f["len"]]) for f in got if f["crc_ok"]}) > 0.9 * len(truth)
    assert (np.diff(got["window"].astype(np.int64)) >= 0).all()          # reference order


# ------------------------------------------------------------------------------------ BLE wideband
def _wb_oracle_frames(oracle_mod, q8):
    return np.concatenate([ble_expected(oracle_mod, q8[c], c) for c in range(40)])


@pytest.mark.parametrize("taps", [384, 768])
def test_ble_wb40_stagewise_parity(Engine, oracle_mod, taps):
    cap = synth.wideband_capture(seconds=0.0085, kind="ble", seed=4000, gap=(200, 2500))
    x = cap.iq[: len(cap.iq) - 24 * 40]                      # ragged: last tile partial
    h = _abi.pfb_prototype(_abi.MODE_BLE_WB40, taps)
    with Engine("ble_wb40", max_samples=len(x), pfb_taps=taps, keep_streams=True) as e:
        got = e.run(x)
        q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0]
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
        bits = e.debug_stage(_abi.STAGE_BLE_BITS)[0]
    # S1: channel streams vs the CPU statement of the channelizer (float64 accumulation)
    yd = oracle_mod.pfb(x, h, [chanplan.ble_channel_bin(c) for c in range(40)])
    rms = np.sqrt(np.mean(np.abs(yd) ** 2))
    assert np.abs(y - yd).max() / rms < CHAN_TOL
    qo = np.clip(np.rint(np.stack([yd.real, yd.imag], -1) * 100.0), -128, 127)
    assert np.abs(q8.astype(int) - qo).max() <= 1
    # S2: frames vs the oracle run on the engine's own quantised streams -- bit exact
    want = _wb_oracle_frames(oracle_mod, q8)
    assert len(want) > 300
    assert_frames_equal(got, want, what=f"wideband {taps} taps")
    # recall against what was transmitted (report-style check, high SNR)
    truth = {(t.channel, bytes(t.data)) for t in cap.truth}
    dec = {(int(f["channel"]), bytes(f["bytes"][:f["len"]])) for f in got if f["crc_ok"]}
    assert len(truth & dec) >= 0.97 * len(truth)
    # the production kernel (no stream stores) must produce the same bits and frames
    with Engine("ble_wb40", max_samples=len(x), pfb_taps=taps) as e:
        got2 = e.run(x)
        bits2 = e.debug_stage(_abi.STAGE_BLE_BITS)[0]
    assert np.array_equal(bits, bits2)
    assert_frames_equal(got2, want, what="production kernel")


def test_ble_wb40_host_pipeline_equals_device_input(Engine):
    """Host input is staged in 32 MiB chunks with the channelizer launched per chunk."""
    import torch
    cap = synth.wideband_capture(seconds=0.06, kind="ble", seed=4100)          # 5.7 M samples = 46 MB: 2 chunks
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        a = e.run(cap.iq)
        b = e.run(torch.from_numpy(cap.iq).cuda())
    assert len(a) > 500
    assert_frames_equal(a, b, what="chunked host input vs device input")


def test_ble_wb40_shards_equal_whole(Engine):
    cap = synth.wideband_capture(seconds=0.025, kind="ble", seed=4200, gap=(200, 3000))
    n_ch = len(cap.iq) // 24
    nw = n_ch // 8192
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        whole = e.run(cap.iq)
        parts = []
        cut = nw // 2
        for w0, w1 in ((0, cut), (cut, nw)):
            lo = max(0, w0 * 8192 - 128) * 24
            hi = min(len(cap.iq), (w1 * 8192 + 2048) * 24)
            parts.append(e.run(cap.iq[lo:hi].copy(), shard=dict(pre_samples=w0 * 8192 * 24 - lo,
                                                               body_samples=(w1 - w0) * 8192 * 24, first_window=w0)))
    got = np.concatenate(parts)
    order = np.lexsort((got["sample_index"], got["window"], got["channel"]))
    assert len(whole) > 300
    assert_frames_equal(got[order], whole, what="2 time shards vs whole")


# ------------------------------------------------------------------------------------ Zigbee narrow band
@pytest.mark.parametrize("segment", [0, 65536])
@pytest.mark.parametrize("seed,esn0", [(2001, 30.0), (2002, 12.0), (2003, 9.0)])
def test_zb_nb_parity(Engine, oracle_mod, seed, esn0, segment):
    cap = synth.zigbee_capture(n=1_000_000, channel=11, seed=seed, esn0_db=esn0)
    with Engine("zb_nb", channel=11, max_samples=len(cap.iq), keep_streams=True, zb_segment=segment) as e:
        got = e.run(cap.iq)
        f = e.debug_stage(_abi.STAGE_ZB_F)[0, 0]
        z = e.debug_stage(_abi.STAGE_ZB_DISC)[0, 0]
        nchips = e.debug_stage(_abi.STAGE_ZB_NCHIPS)
        chips = e.debug_stage(_abi.STAGE_ZB_CHIPS)
    seg, pre = segment or _abi.ZB_SEGMENT_DEFAULT, _abi.ZB_PREHALO_DEFAULT
    fo = oracle_mod.zb_quad_demod(cap.iq)
    assert np.array_equal(f, fo)                                  # same table atan2, same op order: bit exact
    zo = oracle_mod.zb_dc_remove(fo)
    assert np.array_equal(z, zo)                                  # the tracker inside k_zb_rx, stored by the debug build
    # a11 against the published block (north_star: rel err <= 1e-4): the engine's z vs the serial single-pole recurrence
    zs = oracle_mod.zb_dc_remove_serial(fo)
    assert np.abs(z.astype(np.float64) - zs).max() / np.sqrt(np.mean(zs.astype(np.float64) ** 2)) <= 1e-4
    want = oracle_mod.zb_receive(cap.iq, 11, segment=seg, prehalo=pre)
    assert len(want) > 5
    assert_frames_equal(got, want, what=f"zigbee seed {seed}")
    # soft chips of every chain (one per segment): identical count and values, including the step at which
    # a chain stops (post halo, or past its body with the sink searching)
    n_chains = -(-len(zo) // seg)
    assert len(nchips) == n_chains
    for k in range(n_chains):
        lo, hi = k * seg, min(len(zo), (k + 1) * seg)
        _, ck, _ = oracle_mod.zb_chain(zo, max(0, lo - pre), min(len(zo), hi + 16448), lo, hi, want_chips=True, hold=lo - 1024)
        assert nchips[k] == len(ck), (k, nchips[k], len(ck))
        assert np.array_equal(chips[k, : len(ck)], ck), k


def test_zb_nb_lanes_take_several_chains(Engine, oracle_mod, monkeypatch):
    """k_zb_rx hands chains to LANES from a queue inside its window loop.  With the grid capped at one CTA (128 lanes) the 733
    chains of this capture make every lane run five or six chains, restarting at different windows than its neighbours:
    DC-removed stream, frames and the soft chips of every chain must still be the oracle's, bit for bit."""
    monkeypatch.setenv("SNRX_ZB_RX_CTAS", "1")
    cap = synth.zigbee_capture(n=3_000_000, channel=15, seed=2011, esn0_db=14.0)
    with Engine("zb_nb", channel=15, max_samples=len(cap.iq), keep_streams=True) as e:
        got = e.run(cap.iq)
        z = e.debug_stage(_abi.STAGE_ZB_DISC)[0, 0]
        nchips = e.debug_stage(_abi.STAGE_ZB_NCHIPS)
        chips = e.debug_stage(_abi.STAGE_ZB_CHIPS)
    monkeypatch.delenv("SNRX_ZB_RX_CTAS")
    with Engine("zb_nb", channel=15, max_samples=len(cap.iq)) as e:
        free = e.run(cap.iq)
    seg, pre = _abi.ZB_SEGMENT_DEFAULT, _abi.ZB_PREHALO_DEFAULT
    zo = oracle_mod.zb_dc_remove(oracle_mod.zb_quad_demod(cap.iq))
    assert np.array_equal(z, zo)
    want = oracle_mod.zb_receive(cap.iq, 15, segment=seg, prehalo=pre)
    assert len(want) > 20
    assert_frames_equal(got, want, what="one CTA, many chains per lane")
    assert_frames_equal(free, want, what="default grid")
    n_chains = -(-len(zo) // seg)
    assert n_chains > 5 * 128 and len(nchips) == n_chains
    for k in range(0, n_chains, 7):
        lo, hi = k * seg, min(len(zo), (k + 1) * seg)
        _, ck, _ = oracle_mod.zb_chain(zo, max(0, lo - pre), min(len(zo), hi + 16448), lo, hi, want_chips=True, hold=lo - 1024)
        assert nchips[k] == len(ck), (k, nchips[k], len(ck))
        assert np.array_equal(chips[k, : len(ck)], ck), k


def test_zb_chain_order_is_a_scheduling_hint_only(Engine, oracle_mod, monkeypatch):
    """k_zb_order hands the chains that are expected to run long (a burst on the air at the end of their body) to the lanes
    first.  The order must not change a single record: natural order (SNRX_ZB_ORDER=0), longest first (default) and longest
    first on ONE CTA all give the oracle's frames -- on a busy wideband capture (many long chains), on a narrow-band capture
    and on an empty one (no busy block at all)."""
    cap = synth.wideband_capture(seconds=0.03, kind="zigbee", seed=3100, esn0_db=18.0, gap=(400, 6000))
    x = cap.iq
    runs = {}
    for name, env in (("natural", {"SNRX_ZB_ORDER": "0"}), ("longest first", {}), ("longest first, one CTA", {"SNRX_ZB_RX_CTAS": "1"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with Engine("zb_wb16", max_samples=len(x), keep_streams=(name == "natural")) as e:
            runs[name] = e.run(x)
            if name == "natural":
                y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
        for k in env:
            monkeypatch.delenv(k)
    want = np.concatenate([oracle_mod.zb_receive_z(oracle_mod.zb_dc_remove(oracle_mod.zb_quad_demod(y[c])), 11 + c) for c in range(16)])
    assert len(want) > 60
    for name, got in runs.items():
        assert_frames_equal(got, want, what=f"zigbee wideband, chains handed out {name}")
    nb = synth.zigbee_capture(n=1_200_000, channel=18, seed=2012, esn0_db=12.0)
    want_nb = oracle_mod.zb_receive(nb.iq, 18)
    assert len(want_nb) > 8
    for env in ({"SNRX_ZB_ORDER": "0"}, {}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with Engine("zb_nb", channel=18, max_samples=len(nb.iq)) as e:
            assert_frames_equal(e.run(nb.iq), want_nb, what=f"zigbee narrow band {env}")
            assert len(e.run(np.zeros(300_000, np.complex64))) == 0
        for k in env:
            monkeypatch.delenv(k)


def test_zb_nb_batch_and_set_channel(Engine, oracle_mod):
    n = 300_000
    caps = [synth.zigbee_capture(n=n, channel=20, seed=600 + i, esn0_db=20.0, gap=(500, 6000)).iq for i in range(3)]
    with Engine("zb_nb", channel=11, max_samples=n, max_captures=3, zb_segment=32768, zb_prehalo=2048) as e:
        e.set_channel(20)
        got = e.run(np.stack(caps))
    want = []
    for i, c in enumerate(caps):
        f = oracle_mod.zb_receive(c, 20, segment=32768, prehalo=2048)
        f["capture_id"] = i
        want.append(f)
    want = np.concatenate(want)
    assert len(want) > 20
    assert_frames_equal(got, want, what="zigbee batch")
    assert np.array_equal(got["capture_id"], want["capture_id"])


def _zb_shards(n_ch, segment, cuts, pre=None, post=16448 + 64, prehalo=0):
    """[(lo, hi, shard dict)] in channel-rate samples for bodies [cuts[i], cuts[i+1]) segments."""
    from snout_b200 import stream
    if pre is None:
        pre = stream.shard_geometry(0, 1, segment, prehalo)[1]
    out = []
    for s0, s1 in zip(cuts[:-1], cuts[1:]):
        b0, b1 = s0 * segment, min(n_ch, s1 * segment)
        lo = max(0, b0 - pre)
        hi = min(n_ch, b1 + post)
        out.append((lo, hi, dict(pre_samples=b0 - lo, body_samples=b1 - b0, first_window=b0 // 8192)))
    return out


def test_zb_nb_shards_equal_whole(Engine, oracle_mod):
    """Time shards (multi-GPU / streaming unit) reproduce the whole-capture result bit for bit: the DC
    tracker and the chains are defined on absolute grids (oracle/zb_oracle.c)."""
    cap = synth.zigbee_capture(n=1_200_000, channel=17, seed=77, esn0_db=14.0, gap=(500, 9000))
    x = cap.iq
    with Engine("zb_nb", channel=17, max_samples=len(x)) as e:
        whole = e.run(x)
        parts = [e.run(x[lo:hi].copy(), shard=sh) for lo, hi, sh in _zb_shards(len(x), 4096, [0, 80, 190, 293])]
        with pytest.raises(_abi.SnrxError):          # pre halo too short for the tracker memory: refused
            e.run(x[65536 - 4096:].copy(), shard=dict(pre_samples=4096, body_samples=0, first_window=8))
    assert len(whole) > 40
    from snout_b200 import stream
    assert_frames_equal(stream.zb_span_filter(np.concatenate(parts)), whole, what="zigbee: 3 time shards vs whole")
    assert_frames_equal(whole, oracle_mod.zb_receive(x, 17), what="whole vs oracle")


def test_zb_wb16_shards_equal_whole(Engine):
    cap = synth.wideband_capture(seconds=0.05, kind="zigbee", seed=3100, esn0_db=20.0, gap=(400, 5000))
    x = cap.iq
    n_ch = len(x) // 24
    with Engine("zb_wb16", max_samples=len(x), zb_segment=16384, zb_prehalo=4096) as e:
        whole = e.run(x)
        parts = []
        for lo, hi, sh in _zb_shards(n_ch, 16384, [0, 4, 9, 13], prehalo=4096):
            sh = {k: (v * 24 if k != "first_window" else v) for k, v in sh.items()}
            parts.append(e.run(x[lo * 24: hi * 24].copy(), shard=sh))
    from snout_b200 import stream
    got = np.concatenate(parts)
    order = np.lexsort((got["sample_index"], got["window"], got["channel"]))
    assert len(whole) > 60
    assert_frames_equal(stream.zb_span_filter(got[order]), whole, what="zigbee wideband: 3 time shards vs whole")


def test_zb_nb_full_size_config2(Engine, oracle_mod):
    """BASELINE config 2: 1e7 samples of channel 11.  At both segment sizes the decoded frames are exactly the transmitted
    ones (what an unsegmented sequential receiver reports): the span rule removes the CRC-failed syncs of chains that
    start inside a foreign frame (DESIGN.md 4)."""
    cap = synth.zigbee_capture(n=10_000_000, channel=11, seed=2001, esn0_db=30.0)
    truth = [bytes(t.data) for t in cap.truth]
    unsegmented = oracle_mod.zb_receive(cap.iq, 11, segment=1 << 40)
    for seg in (65536, 0):
        with Engine("zb_nb", channel=11, max_samples=10_000_000, zb_segment=seg) as e:
            got = e.run(cap.iq)
        assert_frames_equal(got, oracle_mod.zb_receive(cap.iq, 11, segment=seg or _abi.ZB_SEGMENT_DEFAULT), what=f"config 2, segment {seg}")
        assert [bytes(f["bytes"][:f["len"]]) for f in got] == truth
        assert got["crc_ok"].all()
        assert np.array_equal(got["bytes"], unsegmented["bytes"]) and np.array_equal(got["lqi"], unsegmented["lqi"])


# ------------------------------------------------------------------------------------ Zigbee wideband / mixed
@pytest.mark.parametrize("taps", [384, 768])
def test_zb_wb16_stagewise_parity(Engine, oracle_mod, taps):
    cap = synth.wideband_capture(seconds=0.0125, kind="zigbee", seed=3000, esn0_db=20.0, gap=(400, 5000))
    x = cap.iq[: len(cap.iq) - 24 * 33]
    h = _abi.pfb_prototype(_abi.MODE_ZB_WB16, taps)
    with Engine("zb_wb16", max_samples=len(x), pfb_taps=taps, keep_streams=True, zb_segment=16384, zb_prehalo=2048) as e:
        got = e.run(x)
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
        f = e.debug_stage(_abi.STAGE_ZB_F)[0]
        z = e.debug_stage(_abi.STAGE_ZB_DISC)[0]
    yd = oracle_mod.pfb(x, h, [chanplan.zigbee_channel_bin(c) for c in range(11, 27)])
    assert np.abs(y - yd).max() / np.sqrt(np.mean(np.abs(yd) ** 2)) < CHAN_TOL
    want = []
    for c in range(16):
        fo = oracle_mod.zb_quad_demod(y[c])
        assert np.array_equal(f[c], fo), f"discriminator, channel {11 + c}"
        zo = oracle_mod.zb_dc_remove(fo)
        assert np.array_equal(z[c], zo), f"DC removal, channel {11 + c}"
        want.append(oracle_mod.zb_receive_z(zo, 11 + c, segment=16384, prehalo=2048))
    want = np.concatenate(want)
    assert len(want) > 30
    assert_frames_equal(got, want, what=f"zigbee wideband {taps} taps")
    truth = {(t.channel, bytes(t.data)) for t in cap.truth if t.start + 4400 < len(x) // 24}
    dec = {(int(q["channel"]), bytes(q["bytes"][:q["len"]])) for q in got if q["crc_ok"]}
    assert len(truth & dec) >= 0.95 * len(truth)
    with Engine("zb_wb16", max_samples=len(x), pfb_taps=taps, zb_segment=16384, zb_prehalo=2048) as e:
        assert_frames_equal(e.run(x), want, what="production kernel")


def test_mixed_wb56_equals_separate_engines(Engine):
    cap = synth.wideband_capture(seconds=0.0125, kind="mixed", seed=5000, esn0_db=25.0, gap=(400, 5000))
    x = cap.iq
    with Engine("ble_wb40", max_samples=len(x)) as e:
        a = e.run(x)
    with Engine("zb_wb16", max_samples=len(x)) as e:
        b = e.run(x)
    with Engine("mixed_wb56", max_samples=len(x)) as e:
        m = e.run(x)
    assert len(a) > 50 and len(b) > 4
    assert_frames_equal(m, np.concatenate([a, b]), what="mixed = BLE frames then Zigbee frames")


def test_two_batches_in_flight(Engine):
    caps = [synth.ble_capture(n=200_000, channel=37, seed=700 + i, esn0_db=30, gap=(100, 2000)).iq for i in range(3)]
    with Engine("ble_nb", channel=37, max_samples=200_000) as e:
        ref = [e.run(c) for c in caps]
        e.process(caps[0])
        e.process(caps[1])
        with pytest.raises(_abi.SnrxError):
            e.process(caps[2])                       # a third queued batch is refused, loudly
        r0 = e.poll()
        e.process(caps[2])
        r1 = e.poll()
        r2 = e.poll()
        with pytest.raises(_abi.SnrxError):
            e.poll()                                 # nothing queued
    for got, want in zip((r0, r1, r2), ref):
        assert len(want) > 5
        assert_frames_equal(got, want, what="pipelined batches")


def test_ble_wb40_batch_of_captures(Engine):
    caps = [synth.wideband_capture(seconds=0.0045, kind="ble", seed=4300 + 50 * i, gap=(200, 2500)).iq for i in range(3)]
    with Engine("ble_wb40", max_samples=len(caps[0]), max_captures=3) as e:
        single = []
        for i, c in enumerate(caps):
            f = e.run(c)
            f["capture_id"] = i
            single.append(f)
        got = e.run(np.stack(caps))
    want = np.concatenate(single)
    assert len(want) > 300
    assert_frames_equal(got, want, what="batch of wideband captures")
    assert np.array_equal(got["capture_id"], want["capture_id"])


@pytest.mark.parametrize("mode,kind", [("zb_wb16", "zigbee"), ("mixed_wb56", "mixed")])
def test_wideband_zigbee_and_mixed_batches_of_captures(Engine, mode, kind):
    """The captures of a wideband batch are the y dimension of the channelizer grids (k_pfb_ble, k_pfb_zb_warp) and the outer
    index of the Zigbee chains: a batch of captures gives each capture's own records, and more than 65535 captures per batch
    are refused when the engine is created."""
    caps = [synth.wideband_capture(seconds=0.012, kind=kind, seed=4700 + 31 * i, esn0_db=22.0, gap=(300, 4000)).iq for i in range(2)]
    with Engine(mode, max_samples=len(caps[0]), max_captures=2) as e:
        single = []
        for i, c in enumerate(caps):
            f = e.run(c)
            f["capture_id"] = i
            single.append(f)
        got = e.run(np.stack(caps))
    want = np.concatenate(single)
    assert len(want) > 40 and (want["proto"] == _abi.PROTO_ZIGBEE).sum() > 2     # mixed: most 802.15.4 frames collide with BLE
    assert_frames_equal(_canon_cap(got), _canon_cap(want), what=f"batch of {mode} captures")
    with pytest.raises(_abi.SnrxError):
        Engine(mode, max_samples=24 * 8192, max_captures=65536)


def _canon_cap(fr):
    return fr[np.lexsort((fr["sample_index"], fr["window"], fr["channel"], fr["proto"], fr["capture_id"]))]


# ------------------------------------------------------------------------------------ BASELINE full sizes (configs[2], [3])
def _tile_frames(fr, k, tile_ch, lo_guard=0, hi_guard=0):
    """Frames anchored in tile k (channel-rate tile length tile_ch), positions made tile relative."""
    s = fr["sample_index"]
    sel = fr[(s >= k * tile_ch + lo_guard) & (s < (k + 1) * tile_ch - hi_guard)].copy()
    sel["sample_index"] -= k * tile_ch
    # `window` counts 8192-sample BLE windows / Zigbee chain segments (include/snoutrx.h)
    per = np.where(sel["proto"] == _abi.PROTO_ZIGBEE, _abi.ZB_SEGMENT_DEFAULT, 8192)
    sel["window"] -= ((k * tile_ch) // per).astype(sel["window"].dtype)
    return sel


@pytest.mark.parametrize("mode,kind", [("ble_wb40", "ble"), ("zb_wb16", "zigbee")])
def test_wideband_full_size_time_invariance(Engine, mode, kind):
    """The bench workload at BASELINE size (0.98 s of 96 Msps = 94.4 M samples: a seeded 0.1-s capture tiled x10) checked
    through a size-independent property: the tile length is a multiple of the BLE window / Zigbee segment / DC-block grids
    and of the channelizer's decimation and rotation periods, so every tile that is preceded by a full tile must decode to
    exactly the same records, shifted -- equal to the records of tile 1 of a 3-tile run (whose small-size parity against
    the oracle the stage-wise tests establish).  The last 40 ms of the final tile are excluded (a frame there may run
    past the capture end)."""
    base = synth.wideband_capture(seconds=0.1, kind=kind, seed=4000, esn0_db=25.0).iq
    tile_ch = len(base) // 24
    assert tile_ch % 8192 == 0 and tile_ch % _abi.ZB_IIR_BLOCK == 0
    with Engine(mode, max_samples=10 * len(base), max_frames=1 << 18) as e:
        small = e.run(np.tile(base, 3))
        ref = _tile_frames(small, 1, tile_ch)
        assert len(ref) > (2000 if kind == "ble" else 100)
        big = e.run(np.tile(base, 10))
    assert len(big) > 9 * len(ref)
    for k in range(1, 10):
        guard = 160_000 if k == 9 else 0
        got = _tile_frames(big, k, tile_ch, hi_guard=guard)
        want = ref[ref["sample_index"] < tile_ch - guard]
        key = lambda f: np.lexsort((f["sample_index"], f["window"], f["channel"]))   # noqa: E731
        assert_frames_equal(got[key(got)], want[key(want)], what=f"{mode}: tile {k} of the full-size run vs tile 1 of 3")


def test_zb_reference_pcap_frames_round_trip(Engine, oracle_mod):
    """The 802.15.4 frames of the reference's own test captures (scapy test/pcaps, tests/golden/zb_ref_frames.json) sent
    over the air model and received by the engine: records equal the oracle's and carry exactly those frames."""
    import json
    import os
    from conftest import GOLDEN
    g = json.load(open(os.path.join(GOLDEN, "zb_ref_frames.json")))
    psdus = [bytes.fromhex(h) for h in g["with_fcs"]]
    for h in g["without_fcs"]:
        b = bytes.fromhex(h)
        c = oracle_mod.zb_fcs16(b)
        psdus.append(b + bytes([c & 0xFF, c >> 8]))
    rng = np.random.default_rng(77)
    sig, truth = synth.zb_baseband(1_000_000, 15, rng, gap=(1500, 6000), psdus=psdus)
    x = (sig + synth._awgn(len(sig), rng, 2.0 / 10 ** 2.0)).astype(np.complex64)
    with Engine("zb_nb", channel=15, max_samples=len(x)) as e:
        got = e.run(x)
    assert_frames_equal(got, oracle_mod.zb_receive(x, 15), what="reference pcap frames")
    assert [bytes(f["bytes"][: f["len"]]) for f in got] == [bytes(t.data) for t in truth] and got["crc_ok"].all()
    assert [bytes(f["bytes"][: f["len"]]) for f in got[:55]] == psdus


# ------------------------------------------------------------------------------------ frame exchange (C ABI), one engine
def test_exchange_loopback_world1(Engine):
    """snrx_exchange_* / snrx_allgather with a world of one: the export kernel stores the batch's records (only the
    16-byte pieces in use) and the {count, batch} header into the engine's own receive area; snrx_allgather returns them
    with zeroed tails.  (The multi-rank path over CUDA IPC is exercised by tools/check_multi_gpu.py under torchrun.)"""
    caps = [synth.ble_capture(n=200_000, channel=37, seed=900 + i, esn0_db=30, gap=(100, 1500 + 700 * i)).iq for i in range(3)]
    with Engine("ble_nb", channel=37, max_samples=200_000) as e:
        with pytest.raises(_abi.SnrxError):
            e._xchg_world = 1
            e.allgather(0)                                    # not connected: refused
        e.exchange_connect(e.exchange_create(0, 1, cap_records=1 << 12))
        for k, c in enumerate(caps * 4):                      # 12 batches: the 8 slots are reused
            fr = e.run(c)
            counts, got = e.allgather(e.polled_batch_no, want_frames=True)
            assert counts == [len(fr)] and len(fr) > 20
            assert_frames_equal(got, fr, what=f"loopback batch {k}")
            assert got.tobytes() == fr.tobytes()
        with pytest.raises(_abi.SnrxError):
            e.allgather(e.polled_batch_no + 1, timeout_ms=50)  # a batch nobody has produced: times out
    with Engine("ble_nb", channel=37, max_samples=200_000) as e:
        e.exchange_connect(e.exchange_create(0, 1, cap_records=8))
        fr = e.run(caps[0])
        counts, got = e.allgather(0, want_frames=True)
        assert counts == [len(fr)] and got is None            # more records than the slot holds: counts exact, caller falls back


# ------------------------------------------------------------------------------------ BASELINE configs[4] at full size
def _canon(fr):
    return fr[np.lexsort((fr["sample_index"], fr["window"], fr["channel"], fr["proto"]))]


def test_c5_full_size_time_shards_equal_whole_and_truth(Engine):
    """A 9.81-s 96 Msps mixed BLE + 802.15.4 capture (941.8 M samples, made on the GPU so that every transmitted frame is
    known): (1) cut into ~1-s time shards with the snrx_shard_t halos exactly as dist.plan_job hands them to the ranks of a
    configs[4] job, it yields bit for bit the records of the whole capture processed as ONE batch; (2) what is decoded is what
    was sent: no CRC-ok record carries bytes that were not transmitted on its channel, and the recall of each protocol is
    that of the small-size runs that are checked against the oracle (the two protocols overlap in frequency, so not every
    frame of a mixed capture survives)."""
    from snout_b200 import dist as sdist, stream
    x, truth = synth.wideband_capture_gpu(seconds=0.983, kind="mixed", seed=5000, esn0_db=25.0, repeat=10)
    assert len(x) == 941_752_320 and len(truth) > 250_000       # 10 x 0.983 s (479 windows of 8192 channel samples each)
    with Engine("mixed_wb56", max_samples=len(x), max_frames=1 << 19) as e:
        whole = _canon(e.run(x))
    unit, pre, post = stream.shard_geometry(40, 16)
    parts = []
    with Engine("mixed_wb56", max_samples=(480 * unit + pre + post) * 24, max_frames=1 << 18) as e:
        units = sdist.plan_job(1, len(x), e, units_per_shard=480)
        assert len(units) == 10 and units[1]["pre_samples"] == pre * 24
        for u in units:
            parts.append(e.run(x[u["lo"]: u["hi"]], shard=dict(pre_samples=u["pre_samples"], body_samples=u["body_samples"],
                                                               first_window=u["first_window"])))
    got = _canon(np.concatenate(parts))
    zb = got["proto"] == 2
    got = np.concatenate([stream.zb_span_filter(got[zb]), got[~zb]])
    assert_frames_equal(got, whole, what="configs[4] capture: 10 time shards with halo vs one batch")
    sent = {}
    for t in truth:
        sent.setdefault((t.proto, t.channel), set()).add(bytes(t.data))
    ok = whole[whole["crc_ok"] == 1]
    hits = {2: 0, 3: 0}
    stray = 0
    for f in ok:
        if bytes(f["bytes"][: f["len"]]) in sent[(int(f["proto"]), int(f["channel"]))]:
            hits[int(f["proto"])] += 1
        else:
            stray += 1
    n_sent = {p: sum(1 for t in truth if t.proto == p) for p in (2, 3)}
    stats = dict(records=int(len(whole)), crc_ok=int(len(ok)), sent_ble=n_sent[3], sent_zigbee=n_sent[2], recovered_ble=hits[3],
                 recovered_zigbee=hits[2], stray=stray)
    assert stray <= 3, stats                                  # a CRC-16 lets one random PSDU in 65 536 through
    # 40 BLE and 16 Zigbee transmitters share the band at equal power and frames collide: a 2 MHz O-QPSK frame of up to 4 ms lies
    # over two or three BLE channels that are each busy a quarter of the time, so three quarters of the BLE frames but only
    # one 802.15.4 frame in seven get through with a good FCS (measured: 220 577 / 290 970 and 3 144 / 20 330); the Zigbee
    # receive chain by itself is checked against the oracle and the transmitted frames in test_zb_wb16_stagewise_parity
    assert hits[3] >= 0.70 * n_sent[3] and hits[2] >= 0.12 * n_sent[2], stats


def test_zb_wb16_debug_stream_holds_the_last_sample(Engine, oracle_mod):
    """Found by tools/fuzz_parity.py: when the capture's last channel sample is lane 31 of the last tile (n_out = 31 k + 1) the
    SNRX_STAGE_CHAN_CF32 test stream missed it (the discriminator and the frames were right: they never read that stream)."""
    cap = synth.wideband_capture(seconds=0.01, kind="zigbee", seed=3300, esn0_db=25.0, gap=(400, 4000))
    n_out = (len(cap.iq) // 24 - 40) // 31 * 31 + 1
    x = cap.iq[: n_out * 24]
    with Engine("zb_wb16", max_samples=len(x), keep_streams=True) as e:
        e.run(x)
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
        f = e.debug_stage(_abi.STAGE_ZB_F)[0]
    assert y.shape[1] == n_out and np.all(np.abs(y[:, -1]) > 0)
    for c in range(16):
        assert np.array_equal(f[c], oracle_mod.zb_quad_demod(y[c])), c
