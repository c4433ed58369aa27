"""Per-frame radio metrics (SNRX_F_RF_METRICS, snrx_frame_rf) on the GPU against the float64 restatement
(oracle/rf_oracle.py), and the engine contract around them: frames unchanged, input formats and pointers, shards, lifetime."""
import numpy as np
import pytest

from conftest import assert_frames_equal
from snout_b200 import _abi, stream, synth

pytestmark = pytest.mark.gpu

KEYS = ("sample_index", "capture_id", "frame", "channel", "proto", "valid")
METRICS = ("power_dbfs", "noise_dbfs", "snr_db", "cfo_hz")


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


def _assert_rf_close(got, want, what):
    assert len(got) == len(want), what
    for k in KEYS:
        assert np.array_equal(got[k], want[k]), (what, k)
    for k, tol in (("power_dbfs", 0.01), ("noise_dbfs", 0.01), ("snr_db", 0.02), ("cfo_hz", 100.0)):
        g, w = got[k].astype(np.float64), want[k].astype(np.float64)
        assert np.array_equal(np.isnan(g), np.isnan(w)), (what, k)
        m = ~np.isnan(w)
        d = np.abs(g[m] - w[m])
        if k == "cfo_hz":
            d = np.minimum(d, 4e6 - d)
        assert d.size == 0 or d.max() <= tol, (what, k, float(d.max()), int(np.argmax(d)))


def _assert_rf_identical(got, want, what, keys=KEYS + METRICS):
    assert len(got) == len(want), what
    for k in keys:
        assert np.array_equal(np.ascontiguousarray(got[k]).view(np.uint8), np.ascontiguousarray(want[k]).view(np.uint8)), (what, k)


def _taps(mode, L):
    if mode == "ble_nb" or mode == "zb_nb":
        return {}
    t = {}
    if mode in ("ble_wb40", "mixed_wb56"):
        t["taps_ble"] = _abi.pfb_prototype(_abi.MODE_BLE_WB40, L)
    if mode in ("zb_wb16", "mixed_wb56"):
        t["taps_zb"] = _abi.pfb_prototype(_abi.MODE_ZB_WB16, L)
    return t


def _capture(mode):
    if mode == "ble_nb":
        return synth.ble_capture(n=8192 * 40, channel=37, seed=31, esn0_db=22.0, gap=(200, 3000)).iq, dict(channel=37)
    if mode == "zb_nb":
        return synth.zigbee_capture(n=600_000, channel=15, seed=32, esn0_db=20.0, gap=(1000, 8000)).iq, dict(channel=15)
    kind = {"ble_wb40": "ble", "zb_wb16": "zigbee", "mixed_wb56": "mixed"}[mode]
    secs = {"ble_wb40": 0.01, "zb_wb16": 0.03, "mixed_wb56": 0.02}[mode]
    gap = (200, 3000) if kind == "ble" else (1000, 6000)
    return synth.wideband_capture(seconds=secs, kind=kind, seed=4300, esn0_db=22.0, gap=gap).iq, {}


CASES = [("ble_nb", 0), ("zb_nb", 0)] + [(m, L) for m in ("ble_wb40", "zb_wb16", "mixed_wb56") for L in (384, 768)]


@pytest.mark.parametrize("mode,taps", CASES)
def test_rf_equals_restatement_and_frames_unchanged(Engine, oracle_mod, mode, taps):
    from oracle import rf_oracle
    x, kw = _capture(mode)
    if taps:
        kw["pfb_taps"] = taps
    with Engine(mode, max_samples=len(x), rf_metrics=True, **kw) as e:
        frames = e.run(x)
        rf = e.frame_rf()
    with Engine(mode, max_samples=len(x), **kw) as e:
        plain = e.run(x)
    assert_frames_equal(frames, plain, what=f"{mode}: frames with and without SNRX_F_RF_METRICS")
    assert len(frames) > 10
    want = rf_oracle.frame_rf(x, frames, **_taps(mode, taps or 384))
    _assert_rf_close(rf, want, f"{mode} {taps}")
    assert (rf["valid"] == 7).mean() > 0.9


def test_rf_sc8_device_pointer_and_two_batches(Engine):
    import torch
    cap = synth.ble_capture(n=8192 * 30, channel=38, seed=33, esn0_db=20.0, gap=(200, 3000))
    q8 = np.rint(cap.iq.view(np.float32) * 128).astype(np.int8).reshape(-1, 2)       # the capture lies on the q / 128 grid
    cap2 = synth.ble_capture(n=8192 * 30, channel=38, seed=34, esn0_db=25.0, gap=(200, 3000))
    with Engine("ble_nb", channel=38, max_samples=len(cap.iq), rf_metrics=True) as e:
        e.run(cap.iq)
        ref = e.frame_rf()
        e.run(q8)
        _assert_rf_identical(e.frame_rf(), ref, "sc8 vs cf32 holding q / 128")
        e.run(torch.from_numpy(cap.iq).cuda())
        _assert_rf_identical(e.frame_rf(), ref, "device vs host pointer")
        e.run(torch.from_numpy(q8).cuda())
        _assert_rf_identical(e.frame_rf(), ref, "sc8 device pointer")
        e.run(cap2.iq)
        ref2 = e.frame_rf()
        e.process(cap.iq).process(cap2.iq)                 # two batches in flight keep their own records
        e.poll()
        a = e.frame_rf()
        e.poll()
        b = e.frame_rf()
    assert len(ref) > 10 and len(ref2) > 10
    _assert_rf_identical(a, ref, "first of two in flight")
    _assert_rf_identical(b, ref2, "second of two in flight")

    x, _ = _capture("ble_wb40")
    with Engine("ble_wb40", max_samples=len(x), rf_metrics=True) as e:
        e.run(x)
        ref = e.frame_rf()
        e.run(torch.from_numpy(x).cuda())
        _assert_rf_identical(e.frame_rf(), ref, "wideband: device vs host pointer")


def test_rf_ble_wb40_shards_equal_whole(Engine):
    cap = synth.wideband_capture(seconds=0.025, kind="ble", seed=4200, gap=(200, 3000))
    nw = len(cap.iq) // 24 // 8192
    for taps in (384, 768):
        halo = 128 if taps == 384 else 256
        with Engine("ble_wb40", max_samples=len(cap.iq), pfb_taps=taps, rf_metrics=True) as e:
            whole = e.run(cap.iq)
            rf_whole = e.frame_rf()
            parts, rfs = [], []
            cut = nw // 2
            for w0, w1 in ((0, cut), (cut, nw)):
                lo = max(0, w0 * 8192 - halo) * 24
                hi = min(len(cap.iq), (w1 * 8192 + 2048) * 24)
                parts.append(e.run(cap.iq[lo:hi].copy(), shard=dict(pre_samples=w0 * 8192 * 24 - lo,
                                                                   body_samples=(w1 - w0) * 8192 * 24, first_window=w0)))
                rfs.append(e.frame_rf())
        assert len(whole) > 300 and len(np.concatenate(parts)) == len(whole)
        _assert_rf_identical(stream.rf_of(whole, np.concatenate(rfs)), rf_whole, f"ble_wb40 {taps}: shards vs whole",
                             keys=("sample_index", "capture_id", "channel", "proto", "valid") + METRICS)


def test_rf_ble_nb_shards_equal_whole(Engine):
    cap = synth.ble_capture(n=8192 * 12, channel=37, seed=9, esn0_db=30, gap=(100, 1500))
    with Engine("ble_nb", channel=37, max_samples=8192 * 12, rf_metrics=True) as e:
        whole = e.run(cap.iq)
        rf_whole = e.frame_rf()
        rfs = []
        for w0, w1 in ((0, 5), (5, 9), (9, 12)):
            lo = max(0, w0 * 8192 - 128)
            hi = min(len(cap.iq), w1 * 8192 + 2048)
            e.run(cap.iq[lo:hi].copy(), shard=dict(pre_samples=w0 * 8192 - lo, body_samples=(w1 - w0) * 8192, first_window=w0))
            rfs.append(e.frame_rf())
    assert len(whole) > 20
    _assert_rf_identical(stream.rf_of(whole, np.concatenate(rfs)), rf_whole, "ble_nb: shards vs whole",
                         keys=("sample_index", "capture_id", "channel", "proto", "valid") + METRICS)


def test_rf_zb_wb16_shards_equal_whole(Engine):
    cap = synth.wideband_capture(seconds=0.05, kind="zigbee", seed=3100, esn0_db=20.0, gap=(400, 5000))
    x = cap.iq
    n_ch = len(x) // 24
    seg, prehalo = 16384, 4096
    pre = stream.shard_geometry(0, 1, seg, prehalo)[1]
    with Engine("zb_wb16", max_samples=len(x), zb_segment=seg, zb_prehalo=prehalo, rf_metrics=True) as e:
        whole = e.run(x)
        rf_whole = e.frame_rf()
        rfs = []
        for s0, s1 in ((0, 4), (4, 9), (9, 13)):
            b0, b1 = s0 * seg, min(n_ch, s1 * seg)
            lo, hi = max(0, b0 - pre), min(n_ch, b1 + 16448 + 64)
            e.run(x[lo * 24: hi * 24].copy(), shard=dict(pre_samples=(b0 - lo) * 24, body_samples=(b1 - b0) * 24,
                                                        first_window=b0 // 8192))
            rfs.append(e.frame_rf())
    assert len(whole) > 60
    _assert_rf_identical(stream.rf_of(whole, np.concatenate(rfs)), rf_whole, "zb_wb16: shards vs whole",
                         keys=("sample_index", "capture_id", "channel", "proto", "valid") + METRICS)


def test_rf_768_tap_ble_shard_needs_256_halo_only_with_flag(Engine):
    cap = synth.wideband_capture(seconds=0.01, kind="ble", seed=4201, gap=(200, 3000))
    lo = (8192 - 128) * 24
    shard = dict(pre_samples=128 * 24, body_samples=0, first_window=1)
    with Engine("ble_wb40", max_samples=len(cap.iq), pfb_taps=768) as e:
        e.run(cap.iq[lo:].copy(), shard=shard)
    with Engine("ble_wb40", max_samples=len(cap.iq), pfb_taps=768, rf_metrics=True) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.run(cap.iq[lo:].copy(), shard=shard)
        assert ei.value.code == -1
        e.run(cap.iq[(8192 - 256) * 24:].copy(), shard=dict(pre_samples=256 * 24, body_samples=0, first_window=1))


def test_frame_rf_state_capacity_and_lifetime(Engine):
    from ctypes import byref, c_uint32, c_void_p
    cap = synth.ble_capture(n=8192 * 20, channel=37, seed=35, esn0_db=22.0, gap=(200, 3000))
    cap2 = synth.ble_capture(n=8192 * 20, channel=37, seed=36, esn0_db=22.0, gap=(200, 3000))
    with Engine("ble_nb", channel=37, max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        with pytest.raises(_abi.SnrxError) as ei:
            e.frame_rf()
        assert ei.value.code == -7                           # SNRX_ESTATE: created without SNRX_F_RF_METRICS
    with Engine("ble_nb", channel=37, max_samples=len(cap.iq), rf_metrics=True) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.frame_rf()
        assert ei.value.code == -7                           # nothing polled yet
        frames = e.run(cap.iq)
        n = c_uint32(0)
        out = np.zeros(len(frames), dtype=_abi.RF_DTYPE)
        assert e.lib.snrx_frame_rf(e.handle, None, 0, byref(n)) == 0 and n.value == len(frames)
        assert e.lib.snrx_frame_rf(e.handle, out.ctypes.data_as(c_void_p), len(frames) - 1, byref(n)) == -5   # SNRX_ERANGE
        ref = e.frame_rf()
        # lifetime: the records of a polled batch stay valid until the second-next process, like the summaries'
        e.process(cap.iq).process(cap2.iq)
        e.poll()
        a = e.frame_rf()
        e.process(cap2.iq)                                   # next process after the poll: the records are still there
        _assert_rf_identical(e.frame_rf(), a, "after the next process")
        e.poll()
        e.poll()
    _assert_rf_identical(a, ref, "same input, same records")
