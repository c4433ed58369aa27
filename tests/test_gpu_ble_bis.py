"""snrx_ble_bis on the GPU: equal to oracle/bis_oracle.py on the engine's own bit streams and periodic list, field for field,
with the synthetic truth recovered -- both wideband BLE modes, both prototypes, cf32 and sc8 --; every constructed case of
tests/test_ble_bis.py through the bit-stream hook; the CRC init convention tied to snrx_ble_follow; shards; the calls it
must not disturb; and the state, capacity and lifetime errors."""
from ctypes import byref, c_uint32, c_void_p

import numpy as np
import pytest

from oracle import aux_oracle as ao
from oracle import bis_oracle as bo
from oracle import periodic_oracle as po
from snout_b200 import _abi, chanplan, synth
from test_ble_bis import cases, lists, recovered
from test_gpu_ble_aux import assert_aux_equal, sc8_of
from test_gpu_ble_periodic import assert_sync_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@pytest.fixture(scope="module")
def cap():
    return synth.broadcast_iso_capture(seconds=0.1, seed=9920, esn0_db=25.0, n_bigs=3)


def expected(e, frames, n_out, **kw):
    """(aux, periodic, BIS lists) of the oracles on the engine's own bit streams and records."""
    words = e.debug_stage(_abi.STAGE_BLE_BITS)
    aux = ao.aux_list(words, frames, n_out, **kw)
    sync = po.sync_list(words, aux, n_out, **kw)
    return aux, sync, bo.bis_list(words, sync, n_out, **kw)


@pytest.mark.parametrize("fmt", ["cf32", "sc8"])
@pytest.mark.parametrize("taps", [384, 768])
@pytest.mark.parametrize("mode", ["ble_wb40", "mixed_wb56"])
def test_equals_oracle_and_recovers_truth(Engine, cap, mode, taps, fmt):
    x, scale = (cap.iq, 0.0) if fmt == "cf32" else sc8_of(cap.iq)
    truth = [t for t in cap.meta["bis"] if not t.clash]
    with Engine(mode, max_samples=len(cap.iq), pfb_taps=taps, quant_scale=scale) as e:
        frames = e.run(x)
        aux = e.ble_aux()
        sync = e.ble_periodic()
        bis = e.ble_bis()
        want_aux, want_sync, want = expected(e, frames, len(cap.iq) // 24)
    assert_aux_equal(aux, want_aux, f"{mode} {taps} {fmt} aux")
    assert_sync_equal(sync, want_sync, f"{mode} {taps} {fmt} periodic")
    assert_sync_equal(bis, want, f"{mode} {taps} {fmt}")
    assert {int(p) for p in bis["phy"]} == {0, 1} and (bis["event"] < 0).any()
    assert len(set(bis["source"].tolist())) == 3
    assert recovered(bis, truth) == len(truth), f"{recovered(bis, truth)} of {len(truth)} BIS PDUs"
    assert len(truth) >= 100


@pytest.fixture(scope="module")
def engine(Engine):
    n = max(c.n_out for c in cases())
    with Engine("ble_wb40", max_samples=24 * n, max_captures=3) as e:
        yield e


def test_gpu_equals_oracle_on_every_case(engine):
    for c in cases():
        rec = engine.run_bits(c.words, 24 * c.n_out, shard=c.shard_arg() if (c.shard or c.first_capture) else None)
        want_aux, want_sync = c.lists(rec)
        want = bo.bis_list(c.words, want_sync, c.n_out, **c.geo())
        assert_aux_equal(engine.ble_aux(), want_aux, c.name)
        assert_sync_equal(engine.ble_periodic(), want_sync, c.name)
        got = engine.ble_bis()
        assert_sync_equal(got, want, c.name)
        c.check(got)


def test_follow_finds_the_same_packets(Engine):
    """The CRC init convention against the reference-pinned path: on 1M BISes, follow(AA_n, crc_init_n) decodes every CRC-ok
    BIS PDU whose length byte is below 32 at the same sample (btle_rx's data-channel decoder reads the length as the low 5
    bits of header byte 1)."""
    cap = synth.broadcast_iso_capture(seconds=0.08, seed=9930, esn0_db=25.0, n_bigs=2, phys=(0,), data_len=(0, 24))
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        bis = e.ble_bis()
        compared = 0
        for aa in sorted({int(a) for a in bis["access_addr"]}):
            st = bis[bis["access_addr"] == aa]
            fol = e.follow(aa, int(st["crc_init"][0]))
            for r in st[(st["status"] == bo.OK) & (st["crc_ok"] == 1)]:
                if r["bytes"][1] >= 32:
                    continue
                hit = fol[(fol["sample_index"] == r["sample_index"]) & (fol["channel"] == r["channel"])]
                assert len(hit) == 1 and hit[0]["crc_ok"] == 1, (hex(aa), int(r["event_counter"]), int(r["subevent"]))
                compared += 1
    assert compared >= 20


def test_shards_against_the_whole_capture(Engine, cap):
    n_ch = len(cap.iq) // 24
    n_win = n_ch // 8192
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        whole = e.ble_bis()
        key = {(int(r["access_addr"]), int(r["event_counter"]), int(r["subevent"])): r for r in whole}
        pre, post, compared = 128, 2048, 0
        for w0, w1 in ((0, n_win // 2), (n_win // 2, n_win)):
            a = max(0, w0 * 8192 - pre)
            b = min(n_ch, w1 * 8192 + post)
            shard = dict(pre_samples=(w0 * 8192 - a) * 24, body_samples=(w1 - w0) * 8192 * 24, first_window=w0)
            frames = e.run(cap.iq[a * 24:b * 24], shard=shard)
            got = e.ble_bis()
            _, _, want = expected(e, frames, b - a, first_window=w0, pre_out=w0 * 8192 - a)
            assert_sync_equal(got, want, f"shard {w0}")
            for r in got:                                # a packet found in the shard is the whole capture's
                if r["status"] != bo.OK:
                    continue
                w = key.get((int(r["access_addr"]), int(r["event_counter"]), int(r["subevent"])))
                assert w is not None, (w0, hex(int(r["access_addr"])), int(r["event_counter"]))
                for k in ("sample_index", "status", "crc_ok", "len", "bytes", "phase", "channel", "payload_number"):
                    assert np.array_equal(r[k], w[k]), (k, w0)
                compared += 1
    assert compared >= len(cap.meta["bis"]) // 3, (compared, len(cap.meta["bis"]))


def test_other_calls_are_not_disturbed(Engine, cap):
    def session(with_bis: bool):
        with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
            out = []
            for _ in range(2):
                out.append(e.run(cap.iq))
                if with_bis:
                    e.ble_bis()
                out.append(e.connections())
                out.append(e.ble_aux())
                if with_bis:
                    e.ble_bis()
                out.append(e.ble_coded())
                out.append(e.ble_periodic())
                if with_bis:
                    e.ble_bis()
                out.append(e.follow(chanplan.BLE_ADV_AA, chanplan.BLE_ADV_CRC_INIT))
            e.process(cap.iq)
            if with_bis:
                e.ble_bis()
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
            e.ble_bis()
        assert ei.value.code == -7
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_bis()                                         # nothing polled yet
        assert ei.value.code == -7
        e.run(cap.iq)
        bis = e.ble_bis()
        n = c_uint32(0)
        buf = np.zeros(len(bis) - 1, _abi.BIS_DTYPE)
        rc = e.lib.snrx_ble_bis(e.handle, buf.ctypes.data_as(c_void_p), len(buf), byref(n))
        assert rc == -5 and n.value == len(bis)                 # SNRX_ERANGE, count still reported
        assert e.lib.snrx_ble_bis(e.handle, None, 0, byref(n)) == 0 and n.value == len(bis)
        e.process(cap.iq)
        e.process(cap.iq)                                       # the polled batch's lane is queued again: streams overwritten
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_bis()
        assert ei.value.code == -7
        e.poll(); e.poll()
    # the BIS list is the longest one: EOVERFLOW from it at max_frames + 1, exactly max_frames passes
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        nf = len(e.run(cap.iq))
        na, ns = len(e.ble_aux()), len(e.ble_periodic())
        bis = e.ble_bis()
    assert len(bis) > max(nf, na, ns) + 1, (len(bis), nf, na, ns)
    with Engine("ble_wb40", max_samples=len(cap.iq), max_frames=len(bis) - 1) as e:
        e.run(cap.iq)
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_bis()
        assert ei.value.code == -6 and "BIS" in str(ei.value)
    with Engine("ble_wb40", max_samples=len(cap.iq), max_frames=len(bis)) as e:
        e.run(cap.iq)
        assert e.ble_bis().tobytes() == bis.tobytes()
