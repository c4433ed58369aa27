"""snrx_ble_aux on the GPU: equal to oracle/aux_oracle.py on the engine's own bit streams and polled records, field for field,
and the synthetic truth recovered -- both wideband BLE modes, both prototypes, cf32 and sc8 -- plus multi-capture batches,
shards, the state / capacity / lifetime errors, and the calls it must not disturb."""
from ctypes import byref, c_uint32, c_void_p

import numpy as np
import pytest

from oracle import aux_oracle as ao
from snout_b200 import _abi, chanplan, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@pytest.fixture(scope="module")
def cap():
    return synth.ext_adv_capture(seconds=0.1, seed=9300, esn0_db=25.0, n_events=4, max_chain=2, data_len=(0, 230))


def sc8_of(iq):
    peak = float(np.abs(iq).max())
    q = np.clip(np.rint(iq.view(np.float32).reshape(-1, 2) * (100.0 / peak)), -128, 127).astype(np.int8)
    return q, 128.0 * peak


def expected(e, frames, n_out, **kw):
    return ao.aux_list(e.debug_stage(_abi.STAGE_BLE_BITS), frames, n_out, **kw)


def assert_aux_equal(got, want, what=""):
    assert len(got) == len(want), f"{what}: {len(got)} entries, expected {len(want)}"
    for k in want.dtype.names:
        if not np.array_equal(got[k], want[k]):
            bad = np.nonzero(np.any(np.atleast_2d(got[k] != want[k]).reshape(len(got), -1), axis=1))[0][:5]
            raise AssertionError(f"{what}: field {k} differs at entries {bad.tolist()}")


def recovered(aux, truth, capture_id=0) -> int:
    got = {(int(r["channel"]), int(r["capture_id"]), bytes(r["bytes"][: int(r["len"])]))
           for r in aux if r["status"] == _abi.AUX_OK and r["crc_ok"]}
    return sum((t.channel, capture_id, t.data) in got for t in truth)


@pytest.mark.parametrize("fmt", ["cf32", "sc8"])
@pytest.mark.parametrize("taps", [384, 768])
@pytest.mark.parametrize("mode", ["ble_wb40", "mixed_wb56"])
def test_equals_oracle_and_recovers_truth(Engine, cap, mode, taps, fmt):
    x, scale = (cap.iq, 0.0) if fmt == "cf32" else sc8_of(cap.iq)
    truth = cap.meta["aux"]
    with Engine(mode, max_samples=len(cap.iq), pfb_taps=taps, quant_scale=scale) as e:
        frames = e.run(x)
        aux = e.ble_aux()
        want = expected(e, frames, len(cap.iq) // 24)
    assert_aux_equal(aux, want, f"{mode} {taps} {fmt}")
    assert {int(p) for p in aux["phy"]} == {0, 1} and aux["depth"].max() >= 1
    assert recovered(aux, truth) == len(truth), f"{recovered(aux, truth)} of {len(truth)} aux packets"
    d = {0: [], 1: []}
    for t in truth:                                      # every pointer of the packet found it, at its place (the offset from
        hits = [r for r in aux if r["status"] == _abi.AUX_OK and bytes(r["bytes"][: int(r["len"])]) == t.data]
        assert len(hits) == len(t.parents)               # the nominal AA bit 0 is the filters' delay, the same for every packet)
        d[t.phy] += [int(r["sample_index"]) - t.anchor for r in hits]
    assert all(max(v) - min(v) <= 2 for v in d.values() if v), d


def test_multi_capture_batch_with_stride_padding(Engine, cap):
    other = synth.ext_adv_capture(seconds=0.1, seed=9301, esn0_db=25.0, n_events=4, max_chain=2)
    n = len(cap.iq)
    x = np.zeros((3, n + 48), np.complex64)
    x[0, :n], x[1, :n], x[2, :n] = cap.iq, other.iq, cap.iq
    with Engine("ble_wb40", max_samples=n, max_captures=3) as e:
        frames = e.run(x, n_samples=n, stride=n + 48)
        aux = e.ble_aux()
        assert_aux_equal(aux, expected(e, frames, n // 24), "3 captures")
        single = e.run(cap.iq)
        one = e.ble_aux()
    assert recovered(aux, cap.meta["aux"], 0) == len(cap.meta["aux"])
    assert recovered(aux, other.meta["aux"], 1) == len(other.meta["aux"])
    assert recovered(aux, cap.meta["aux"], 2) == len(cap.meta["aux"])
    a0 = aux[aux["capture_id"] == 0]
    for k in ("sample_index", "win_lo", "win_hi", "status", "crc_ok", "len", "bytes", "channel", "phy", "depth"):
        assert np.array_equal(a0[k], one[k]), k
    assert len(single) > 0


def test_shards_against_the_whole_capture(Engine, cap):
    n_ch = len(cap.iq) // 24
    n_win = n_ch // 8192
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        whole = e.ble_aux()
        key = {(int(r["depth"]), int(r["win_lo"]), int(r["win_hi"]), int(r["channel"]), int(r["phy"])): r for r in whole}
        pre, post, compared = 128, 2048, 0
        for w0, w1 in ((0, n_win // 2), (n_win // 2, n_win)):
            a = max(0, w0 * 8192 - pre)
            b = min(n_ch, w1 * 8192 + post)
            shard = dict(pre_samples=(w0 * 8192 - a) * 24, body_samples=(w1 - w0) * 8192 * 24, first_window=w0)
            frames = e.run(cap.iq[a * 24:b * 24], shard=shard)
            got = e.ble_aux()
            assert_aux_equal(got, expected(e, frames, b - a, first_window=w0, pre_out=w0 * 8192 - a), f"shard {w0}")
            for r in got:
                if r["status"] in (_abi.AUX_OUTSIDE, _abi.AUX_TRUNCATED):      # reaches past this shard's buffer
                    continue
                w = key[(int(r["depth"]), int(r["win_lo"]), int(r["win_hi"]), int(r["channel"]), int(r["phy"]))]
                for k in ("sample_index", "status", "crc_ok", "len", "bytes", "phase"):
                    assert np.array_equal(r[k], w[k]), (k, w0)
                compared += 1
    assert compared >= len(cap.meta["aux"])


def test_other_calls_are_not_disturbed(Engine, cap):
    def session(with_aux: bool):
        with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
            out = []
            for _ in range(2):
                out.append(e.run(cap.iq))
                if with_aux:
                    e.ble_aux()
                out.append(e.connections())
                if with_aux:
                    e.ble_aux()
                out.append(e.follow(chanplan.BLE_ADV_AA, chanplan.BLE_ADV_CRC_INIT))
            e.process(cap.iq)
            out.append(e.poll())
            return out
    a, b = session(False), session(True)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    assert sum(len(x) for x in a) > 0


def test_state_capacity_and_lifetime_errors(Engine, cap):
    with Engine("ble_nb", channel=37, max_samples=100_000) as e:
        e.run(np.zeros(100_000, np.complex64))
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_aux()
        assert ei.value.code == -7
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_aux()                                         # nothing polled yet
        assert ei.value.code == -7
        frames = e.run(cap.iq)
        aux = e.ble_aux()
        n = c_uint32(0)
        buf = np.zeros(len(aux) - 1, _abi.AUX_DTYPE)
        rc = e.lib.snrx_ble_aux(e.handle, buf.ctypes.data_as(c_void_p), len(buf), byref(n))
        assert rc == -5 and n.value == len(aux)                 # SNRX_ERANGE, count still reported
        assert e.lib.snrx_ble_aux(e.handle, None, 0, byref(n)) == 0 and n.value == len(aux)
        e.process(cap.iq)
        e.process(cap.iq)                                       # the polled batch's lane is queued again: streams overwritten
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_aux()
        assert ei.value.code == -7
        e.poll(); e.poll()
    # 2M-only aux packets are not decoded as data-channel frames, so a chain gives more entries than the batch has records
    cap2 = synth.ext_adv_capture(seconds=0.1, seed=9302, esn0_db=25.0, n_events=4, max_chain=3, phys=(1,))
    with Engine("ble_wb40", max_samples=len(cap2.iq)) as e:
        nf = len(e.run(cap2.iq))
        aux = e.ble_aux()
    assert len(aux) > nf
    with Engine("ble_wb40", max_samples=len(cap2.iq), max_frames=nf) as e:
        assert len(e.run(cap2.iq)) == nf
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_aux()
        assert ei.value.code == -6                              # SNRX_EOVERFLOW
    with Engine("ble_wb40", max_samples=len(cap2.iq), max_frames=len(aux)) as e:
        e.run(cap2.iq)
        assert e.ble_aux().tobytes() == aux.tobytes()
