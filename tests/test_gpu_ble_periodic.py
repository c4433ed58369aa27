"""snrx_ble_periodic on the GPU: equal to oracle/periodic_oracle.py on the engine's own bit streams and aux list, field for
field, with the synthetic truth recovered -- both wideband BLE modes, both prototypes, cf32 and sc8 --; every constructed
case of tests/test_ble_periodic.py through the bit-stream hook; the CRCInit convention tied to snrx_ble_follow; shards; the
calls it must not disturb; and the state, capacity and lifetime errors."""
from ctypes import byref, c_uint32, c_void_p

import numpy as np
import pytest

from oracle import aux_oracle as ao
from oracle import periodic_oracle as po
from snout_b200 import _abi, chanplan, synth
from test_ble_periodic import cases, recovered
from test_gpu_ble_aux import assert_aux_equal, sc8_of

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@pytest.fixture(scope="module")
def cap():
    return synth.periodic_adv_capture(seconds=0.1, seed=9720, esn0_db=25.0, n_trains=4, intervals=(6, 30))


def expected(e, frames, n_out, **kw):
    """(aux list, periodic list) of the oracles on the engine's own bit streams and records."""
    words = e.debug_stage(_abi.STAGE_BLE_BITS)
    aux = ao.aux_list(words, frames, n_out, **kw)
    return aux, po.sync_list(words, aux, n_out, **kw)


def assert_sync_equal(got, want, what=""):
    assert len(got) == len(want), f"{what}: {len(got)} entries, expected {len(want)}"
    for k in want.dtype.names:
        if not np.array_equal(got[k], want[k]):
            bad = np.nonzero(np.any(np.atleast_2d(got[k] != want[k]).reshape(len(got), -1), axis=1))[0][:5]
            raise AssertionError(f"{what}: field {k} differs at entries {bad.tolist()}")


@pytest.mark.parametrize("fmt", ["cf32", "sc8"])
@pytest.mark.parametrize("taps", [384, 768])
@pytest.mark.parametrize("mode", ["ble_wb40", "mixed_wb56"])
def test_equals_oracle_and_recovers_truth(Engine, cap, mode, taps, fmt):
    x, scale = (cap.iq, 0.0) if fmt == "cf32" else sc8_of(cap.iq)
    truth = [t for t in cap.meta["sync"] if not t.clash]
    with Engine(mode, max_samples=len(cap.iq), pfb_taps=taps, quant_scale=scale) as e:
        frames = e.run(x)
        aux = e.ble_aux()
        sync = e.ble_periodic()
        want_aux, want = expected(e, frames, len(cap.iq) // 24)
    assert_aux_equal(aux, want_aux, f"{mode} {taps} {fmt} aux")
    assert_sync_equal(sync, want, f"{mode} {taps} {fmt}")
    assert {int(p) for p in sync["phy"]} == {0, 1} and (sync["event"] < 0).any()
    assert len({int(a) for a in sync["access_addr"]}) == 4
    assert recovered(sync, truth) == len(truth), f"{recovered(sync, truth)} of {len(truth)} AUX_SYNC_INDs"
    assert len(truth) >= 20 and {t.counter for t in truth} >= {65535, 0}


@pytest.fixture(scope="module")
def engine(Engine):
    n = max(c.n_out for c in cases())
    with Engine("ble_wb40", max_samples=24 * n, max_captures=3) as e:
        yield e


def test_gpu_equals_oracle_on_every_case(engine):
    for c in cases():
        rec = engine.run_bits(c.words, 24 * c.n_out, shard=c.shard_arg() if (c.shard or c.first_capture) else None)
        for cap_i, ch, s in c.spots:
            assert ((rec["sample_index"] == s) & (rec["channel"] == ch) & (rec["crc_ok"] == 1)
                    & (rec["capture_id"] == c.first_capture + cap_i)).any(), (c.name, s)
        aux = engine.ble_aux()
        want_aux, want = c.lists(rec)
        assert_aux_equal(aux, want_aux, c.name)
        got = engine.ble_periodic()
        assert_sync_equal(got, want, c.name)
        c.check(got)


def test_follow_finds_the_same_packets(Engine):
    """The CRCInit convention against the reference-pinned path: on 1M trains, follow(train AA, train crc_init) decodes every
    CRC-ok AUX_SYNC_IND whose length byte is below 32 at the same sample.  btle_rx's data-channel decoder reads the length as
    the low 5 bits of header byte 1 (and at most 37 payload bytes), so only those lengths are read alike by both."""
    cap = synth.periodic_adv_capture(seconds=0.08, seed=9730, esn0_db=25.0, n_trains=3, phys=(0,), intervals=(6, 10),
                                      data_len=(0, 24), big_info=False)
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        sync = e.ble_periodic()
        compared = 0
        for aa in sorted({int(a) for a in sync["access_addr"]}):
            tr = sync[sync["access_addr"] == aa]
            fol = e.follow(aa, int(tr["crc_init"][0]))
            for r in tr[(tr["status"] == po.OK) & (tr["crc_ok"] == 1)]:
                if r["bytes"][1] >= 32:
                    continue
                hit = fol[(fol["sample_index"] == r["sample_index"]) & (fol["channel"] == r["channel"])]
                assert len(hit) == 1 and hit[0]["crc_ok"] == 1, (hex(aa), int(r["event_counter"]))
                compared += 1
    assert compared >= 10


def test_shards_against_the_whole_capture(Engine, cap):
    n_ch = len(cap.iq) // 24
    n_win = n_ch // 8192
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        whole = e.ble_periodic()
        key = {(int(r["access_addr"]), int(r["event_counter"])): r for r in whole}
        pre, post, compared = 128, 2048, 0
        for w0, w1 in ((0, n_win // 2), (n_win // 2, n_win)):
            a = max(0, w0 * 8192 - pre)
            b = min(n_ch, w1 * 8192 + post)
            shard = dict(pre_samples=(w0 * 8192 - a) * 24, body_samples=(w1 - w0) * 8192 * 24, first_window=w0)
            frames = e.run(cap.iq[a * 24:b * 24], shard=shard)
            got = e.ble_periodic()
            aux = e.ble_aux()
            want_aux, want = expected(e, frames, b - a, first_window=w0, pre_out=w0 * 8192 - a)
            assert_aux_equal(aux, want_aux, f"shard {w0} aux")
            assert_sync_equal(got, want, f"shard {w0}")
            for r in got:                                # a packet found in the shard is the whole capture's
                if r["status"] != po.OK:
                    continue
                w = key.get((int(r["access_addr"]), int(r["event_counter"])))
                assert w is not None, (w0, hex(int(r["access_addr"])), int(r["event_counter"]))
                for k in ("sample_index", "status", "crc_ok", "len", "bytes", "phase", "channel"):
                    assert np.array_equal(r[k], w[k]), (k, w0)
                compared += 1
    # each shard predicts its trains from its own AUX_ADV_INDs: a train without one in a shard is not listed there
    assert compared >= len(cap.meta["sync"]) // 2, (compared, len(cap.meta["sync"]))


def test_other_calls_are_not_disturbed(Engine, cap):
    def session(with_sync: bool):
        with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
            out = []
            for _ in range(2):
                out.append(e.run(cap.iq))
                if with_sync:
                    e.ble_periodic()
                out.append(e.connections())
                out.append(e.ble_aux())
                if with_sync:
                    e.ble_periodic()
                out.append(e.ble_coded())
                out.append(e.follow(chanplan.BLE_ADV_AA, chanplan.BLE_ADV_CRC_INIT))
            e.process(cap.iq)
            if with_sync:
                e.ble_periodic()
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
            e.ble_periodic()
        assert ei.value.code == -7
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_periodic()                                    # nothing polled yet
        assert ei.value.code == -7
        frames = e.run(cap.iq)
        sync = e.ble_periodic()
        n = c_uint32(0)
        buf = np.zeros(len(sync) - 1, _abi.SYNC_DTYPE)
        rc = e.lib.snrx_ble_periodic(e.handle, buf.ctypes.data_as(c_void_p), len(buf), byref(n))
        assert rc == -5 and n.value == len(sync)                # SNRX_ERANGE, count still reported
        assert e.lib.snrx_ble_periodic(e.handle, None, 0, byref(n)) == 0 and n.value == len(sync)
        e.process(cap.iq)
        e.process(cap.iq)                                       # the polled batch's lane is queued again: streams overwritten
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_periodic()
        assert ei.value.code == -7
        e.poll(); e.poll()
    # few advertising events, many periodic events: the periodic list is the longest one
    cap2 = synth.periodic_adv_capture(seconds=0.1, seed=9740, esn0_db=25.0, n_trains=4, intervals=(6, 6),
                                      adv_interval=(300_000, 300_000))
    with Engine("ble_wb40", max_samples=len(cap2.iq)) as e:
        nf = len(e.run(cap2.iq))
        na = len(e.ble_aux())
        sync = e.ble_periodic()
    assert len(sync) > max(nf, na) + 1, (len(sync), nf, na)
    with Engine("ble_wb40", max_samples=len(cap2.iq), max_frames=len(sync) - 1) as e:
        e.run(cap2.iq)
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_periodic()
        assert ei.value.code == -6                              # SNRX_EOVERFLOW at max_frames + 1
    with Engine("ble_wb40", max_samples=len(cap2.iq), max_frames=len(sync)) as e:
        e.run(cap2.iq)
        assert e.ble_periodic().tobytes() == sync.tobytes()
    # 2M-only chains: more aux entries than records, so the aux rounds refuse first
    cap3 = synth.ext_adv_capture(seconds=0.1, seed=9302, esn0_db=25.0, n_events=4, max_chain=3, phys=(1,))
    with Engine("ble_wb40", max_samples=len(cap3.iq)) as e:
        nf = len(e.run(cap3.iq))
        na = len(e.ble_aux())
        assert len(e.ble_periodic()) == 0
    assert na > nf
    with Engine("ble_wb40", max_samples=len(cap3.iq), max_frames=nf) as e:
        e.run(cap3.iq)
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_periodic()
        assert ei.value.code == -6
