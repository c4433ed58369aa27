"""k_zb_rx, k_zb_span_filter and k_zb_gather on constructed chip streams (tests/zb_chips.py): every case through the
narrow-band engine equals the oracle field for field, in the production build and in the keep_streams build, whose
DC-removed stream and soft chips equal the oracle's bit for bit chain by chain -- on the drift cases that is what pins the
tracker's catch-up and pause windows.  Also: one CTA with chains handed out in natural order, a time shard with frames on
its body edges, and max_frames at the frame count and one below, in zb_nb and in mixed_wb56 (where the Zigbee records
follow the BLE ones)."""
import functools

import numpy as np
import pytest

import zb_chips as Z
from conftest import assert_frames_equal
from snout_b200 import _abi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@functools.lru_cache(maxsize=None)
def _cases():
    return {c.name: c for c in Z.cases()}


NAMES = [c.name for c in Z.cases()]


def _engine(Engine, case, **kw):
    caps = case.captures
    return Engine("zb_nb", channel=Z.CHANNEL, max_samples=caps.shape[1], max_captures=len(caps), zb_threshold=case.threshold,
                  zb_segment=case.segment, zb_prehalo=case.prehalo, **kw)


def _check_streams(oracle_mod, case, z, nchips, chips):
    n_seg = -(-case.captures.shape[1] // case.segment)
    assert len(nchips) == n_seg * len(case.captures)
    for i, x in enumerate(case.captures):
        zo = oracle_mod.zb_dc_remove(oracle_mod.zb_quad_demod(x))
        assert np.array_equal(z[i, 0], zo), (case.name, i)
        for c, (lo, hi, begin, end) in enumerate(Z.chain_geometry(len(zo), case.segment, case.prehalo)):
            _, ck, _ = oracle_mod.zb_chain(zo, begin, end, lo, hi, threshold=case.threshold, want_chips=True, hold=lo - Z.SINK_LEAD)
            k = i * n_seg + c
            assert nchips[k] == len(ck), (case.name, i, c, nchips[k], len(ck))
            assert np.array_equal(chips[k, :len(ck)], ck), (case.name, i, c)


@pytest.mark.parametrize("name", NAMES)
def test_case_on_the_gpu(Engine, oracle_mod, name):
    case = _cases()[name]
    want = Z.oracle_frames(oracle_mod, case)
    with _engine(Engine, case) as e:
        got = e.run(case.iq)
    assert_frames_equal(got, want, what=f"{name}, production build")
    assert np.array_equal(got["capture_id"], want["capture_id"])
    with _engine(Engine, case, keep_streams=True) as e:
        kept = e.run(case.iq)
        z = e.debug_stage(_abi.STAGE_ZB_DISC)
        nchips = e.debug_stage(_abi.STAGE_ZB_NCHIPS)
        chips = e.debug_stage(_abi.STAGE_ZB_CHIPS)
    assert_frames_equal(kept, want, what=f"{name}, keep_streams build")
    _check_streams(oracle_mod, case, z, nchips, chips)


def test_drift_on_one_cta_in_natural_order(Engine, oracle_mod, monkeypatch):
    """Every lane runs many chains, restarting its tracker at other windows than its neighbours, while the drift makes a
    third of the windows catch up and a third pause."""
    monkeypatch.setenv("SNRX_ZB_RX_CTAS", "1")
    monkeypatch.setenv("SNRX_ZB_ORDER", "0")
    case = _cases()["drift_+0.003"]
    x = np.tile(case.iq, (3, 1))
    batch = Z.Case("drift batch", x, None, "", case.threshold, 16384, case.prehalo)
    with _engine(Engine, batch, keep_streams=True) as e:
        got = e.run(x)
        z = e.debug_stage(_abi.STAGE_ZB_DISC)
        nchips = e.debug_stage(_abi.STAGE_ZB_NCHIPS)
        chips = e.debug_stage(_abi.STAGE_ZB_CHIPS)
    assert_frames_equal(got, Z.oracle_frames(oracle_mod, batch), what="one CTA, natural order")
    _check_streams(oracle_mod, batch, z, nchips, chips)


def test_shard_body_edges(Engine, oracle_mod):
    """A time shard of four captures (first capture id 5) whose frames sync at b0 - 1, b0, b1 - 1 and b1 of the shard body:
    only the two inside it are reported, with the whole capture's sample index, window and the shard's capture ids."""
    xs, targets, shard, lo = Z.shard_edge_captures()
    part = np.ascontiguousarray(xs[:, lo:])
    want = []
    w0, w1 = shard["first_window"] * 8192 // Z.SEGMENT, (shard["first_window"] * 8192 + shard["body_samples"]) // Z.SEGMENT
    for i, x in enumerate(xs):
        f = oracle_mod.zb_receive(x, Z.CHANNEL)
        f = f[(f["window"] >= w0) & (f["window"] < w1)]
        f["capture_id"] = shard["first_capture_id"] + i
        want.append(f)
    want = np.concatenate(want)
    assert list(want["sample_index"]) == list(targets[1:3])
    with Engine("zb_nb", channel=Z.CHANNEL, max_samples=part.shape[1], max_captures=len(part)) as e:
        got = e.run(part, shard=shard)
    assert_frames_equal(got, want, what="shard body edges")
    assert np.array_equal(got["capture_id"], want["capture_id"])


def test_max_frames_at_the_zigbee_frame_count(Engine, oracle_mod):
    """zb_nb: max_frames equal to the record count passes; one less fails the batch with SNRX_EOVERFLOW, and the next batch
    of the same engine is complete."""
    case = _cases()["phr_edges"]
    want = Z.oracle_frames(oracle_mod, case)
    assert len(want) == 4
    with _engine(Engine, case, max_frames=4) as e:
        assert_frames_equal(e.run(case.iq), want, what="max_frames = 4")
    with _engine(Engine, case, max_frames=3) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.run(case.iq)
        assert ei.value.code == -6
        small = _cases()["thr10_decode"]
        x = np.zeros(len(case.iq), np.complex64)
        x[:len(small.iq)] = small.iq
        assert_frames_equal(e.run(x), oracle_mod.zb_receive(x, Z.CHANNEL), what="the batch after an overflow")


def test_max_frames_in_mixed_wb56(Engine):
    """mixed_wb56 gathers the Zigbee records after the BLE ones: max_frames at the total count passes, one below fails with
    SNRX_EOVERFLOW, and the next batch is complete."""
    cap = synth.wideband_capture(seconds=0.0125, kind="mixed", seed=5000, esn0_db=25.0, gap=(400, 5000))
    half = cap.iq[: len(cap.iq) // 2 // 24 * 24]
    with Engine("mixed_wb56", max_samples=len(cap.iq)) as e:
        full = e.run(cap.iq)
        want_half = e.run(half)
    n = len(full)
    assert (full["proto"] == _abi.PROTO_ZIGBEE).sum() > 5 and (full["proto"] != _abi.PROTO_ZIGBEE).sum() > 5
    with Engine("mixed_wb56", max_samples=len(cap.iq), max_frames=n) as e:
        assert_frames_equal(e.run(cap.iq), full, what="max_frames = frame count")
    with Engine("mixed_wb56", max_samples=len(cap.iq), max_frames=n - 1) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.run(cap.iq)
        assert ei.value.code == -6
        assert len(want_half) < n - 1
        assert_frames_equal(e.run(half), want_half, what="the batch after an overflow")
