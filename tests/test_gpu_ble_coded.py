"""snrx_ble_coded on the GPU: equal to oracle/coded_oracle.py on the engine's own bit streams, field for field, and the
synthetic truth recovered -- both wideband BLE modes, both prototypes, cf32 and sc8 -- plus multi-capture batches, shards,
the state / capacity / lifetime errors, the calls it must not disturb, and the primaries a dense legacy capture gives."""
from ctypes import byref, c_uint32, c_void_p

import numpy as np
import pytest

from oracle import coded_oracle as co
from snout_b200 import _abi, chanplan, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@pytest.fixture(scope="module")
def cap():
    return synth.coded_adv_capture(seconds=0.15, seed=9700, esn0_db=25.0, n_events=4, max_chain=2)


def sc8_of(iq):
    peak = float(np.abs(iq).max())
    q = np.clip(np.rint(iq.view(np.float32).reshape(-1, 2) * (100.0 / peak)), -128, 127).astype(np.int8)
    return q, 128.0 * peak


def expected(e, n_out, **kw):
    return co.coded_list(e.debug_stage(_abi.STAGE_BLE_BITS), n_out, **kw)


def assert_coded_equal(got, want, what=""):
    assert len(got) == len(want), f"{what}: {len(got)} entries, expected {len(want)}"
    for k in want.dtype.names:
        if not np.array_equal(got[k], want[k]):
            bad = np.nonzero(np.any(np.atleast_2d(got[k] != want[k]).reshape(len(got), -1), axis=1))[0][:5]
            raise AssertionError(f"{what}: field {k} differs at entries {bad.tolist()}")


def recovered(lst, truth, capture_id=0) -> int:
    got = {(int(r["channel"]), int(r["capture_id"]), bytes(r["bytes"][: int(r["len"])]))
           for r in lst if r["status"] == _abi.AUX_OK and r["crc_ok"]}
    return sum((t.channel, capture_id, t.data) in got for t in truth)


@pytest.mark.parametrize("fmt", ["cf32", "sc8"])
@pytest.mark.parametrize("taps", [384, 768])
@pytest.mark.parametrize("mode", ["ble_wb40", "mixed_wb56"])
def test_equals_oracle_and_recovers_truth(Engine, cap, mode, taps, fmt):
    x, scale = (cap.iq, 0.0) if fmt == "cf32" else sc8_of(cap.iq)
    truth = cap.meta["coded"]
    with Engine(mode, max_samples=len(cap.iq), pfb_taps=taps, quant_scale=scale) as e:
        e.run(x)
        got = e.ble_coded()
        want = expected(e, len(cap.iq) // 24)
    assert_coded_equal(got, want, f"{mode} {taps} {fmt}")
    assert {int(t.phy) for t in truth} <= {int(p) for p in got["phy"]} and got["depth"].max() == max(t.depth for t in truth)
    assert recovered(got, truth) == len(truth), f"{recovered(got, truth)} of {len(truth)} packets"
    prim = got[got["depth"] == 0]
    ok = prim[(prim["status"] == _abi.AUX_OK) & (prim["crc_ok"] == 1)]
    assert len(ok) == sum(t.depth == 0 for t in truth)
    d = [int(r["sample_index"]) - t.anchor for t in truth if t.depth == 0 for r in ok if bytes(r["bytes"][: int(r["len"])]) == t.data
         and r["channel"] == t.channel]
    assert max(d) - min(d) <= 2, d                     # every primary at its place (the filters' delay within a sample)
    assert set(ok["ci"]) <= {0, 1} and {int(r["ci"]) for r in ok} == {0 if t.s == 8 else 1 for t in truth if t.depth == 0}


def test_multi_capture_batch_with_stride_padding(Engine, cap):
    other = synth.coded_adv_capture(seconds=0.15, seed=9701, esn0_db=25.0, n_events=4, max_chain=2)
    n = len(cap.iq)
    x = np.zeros((3, n + 48), np.complex64)
    x[0, :n], x[1, :n], x[2, :n] = cap.iq, other.iq, cap.iq
    with Engine("ble_wb40", max_samples=n, max_captures=3) as e:
        e.run(x, n_samples=n, stride=n + 48)
        got = e.ble_coded()
        assert_coded_equal(got, expected(e, n // 24), "3 captures")
        e.run(cap.iq)
        one = e.ble_coded()
    assert recovered(got, cap.meta["coded"], 0) == len(cap.meta["coded"])
    assert recovered(got, other.meta["coded"], 1) == len(other.meta["coded"])
    assert recovered(got, cap.meta["coded"], 2) == len(cap.meta["coded"])
    a0 = got[got["capture_id"] == 0]
    for k in ("sample_index", "win_lo", "win_hi", "status", "crc_ok", "len", "bytes", "channel", "phy", "depth", "ci",
              "aa_errors", "metric"):
        assert np.array_equal(a0[k], one[k]), k


@pytest.mark.parametrize("post", [2048, 67_840 + 2048])
def test_shards_against_the_whole_capture(Engine, cap, post):
    """Every shard equals the oracle on its own buffer.  Its entries that are neither TRUNCATED nor OUTSIDE equal the whole
    capture's, each whole-capture entry is matched by one shard at most, and every primary by exactly one: with a post halo
    of 67 840 samples or more, no primary of a body is TRUNCATED unless it is so in the whole capture."""
    n_ch = len(cap.iq) // 24
    n_win = n_ch // 8192
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        whole = e.ble_coded()
        key = lambda r: (int(r["depth"]), int(r["win_lo"]), int(r["win_hi"]), int(r["channel"]), int(r["phy"]))  # noqa: E731
        index = {key(r): k for k, r in enumerate(whole)}
        assert len(index) == len(whole)
        matched = np.zeros(len(whole), int)
        pre, cut = 128, 0
        for w0, w1 in ((0, n_win // 3), (n_win // 3, 2 * n_win // 3), (2 * n_win // 3, n_win)):
            a = max(0, w0 * 8192 - pre)
            b = min(n_ch, w1 * 8192 + post)
            shard = dict(pre_samples=(w0 * 8192 - a) * 24, body_samples=(w1 - w0) * 8192 * 24, first_window=w0)
            e.run(cap.iq[a * 24:b * 24], shard=shard)
            got = e.ble_coded()
            assert_coded_equal(got, expected(e, b - a, first_window=w0, pre_out=w0 * 8192 - a, n_windows=w1 - w0), f"shard {w0}")
            for r in got:
                k = index[key(r)]
                w = whole[k]
                if r["status"] in (_abi.AUX_OUTSIDE, _abi.AUX_TRUNCATED) and w["status"] != r["status"]:
                    cut += 1                                  # reaches past this shard's buffer
                    assert r["depth"] > 0 or post < 67_840, (w0, int(r["sample_index"]))
                    continue
                for f in ("sample_index", "status", "crc_ok", "len", "bytes", "phase", "ci", "aa_errors", "metric"):
                    assert np.array_equal(r[f], w[f]), (f, w0)
                matched[k] += 1
    prim = whole["depth"] == 0
    assert matched.max() <= 1
    if post > 67_840:
        assert (matched[prim] == 1).all()
    print(f"post-halo {post}: {int(matched.sum())} of {len(whole)} entries equal to the whole capture's, {cut} cut by the buffer")


def test_other_calls_are_not_disturbed(Engine, cap):
    x = cap.iq + legacy_capture(seconds=0.15)                 # Long Range events over legacy traffic
    assert len(x) == len(cap.iq)

    def session(with_coded: bool):
        with Engine("ble_wb40", max_samples=len(x)) as e:
            out = []
            for _ in range(2):
                out.append(e.run(x))
                if with_coded:
                    e.ble_coded()
                out.append(e.connections())
                out.append(e.ble_aux())
                if with_coded:
                    e.ble_coded()
                out.append(e.follow(chanplan.BLE_ADV_AA, chanplan.BLE_ADV_CRC_INIT))
            e.process(x)
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
            e.ble_coded()
        assert ei.value.code == -7
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_coded()                                       # nothing polled yet
        assert ei.value.code == -7
        e.run(cap.iq)
        lst = e.ble_coded()
        n = c_uint32(0)
        buf = np.zeros(len(lst) - 1, _abi.CODED_DTYPE)
        rc = e.lib.snrx_ble_coded(e.handle, buf.ctypes.data_as(c_void_p), len(buf), byref(n))
        assert rc == -5 and n.value == len(lst)                 # SNRX_ERANGE, count still reported
        assert e.lib.snrx_ble_coded(e.handle, None, 0, byref(n)) == 0 and n.value == len(lst)
        e.process(cap.iq)
        e.process(cap.iq)                                       # the polled batch's lane is queued again: streams overwritten
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_coded()
        assert ei.value.code == -7
        e.poll(); e.poll()
    # Coded packets are not legacy records: the list is longer than the batch's record count
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        nf = len(e.run(cap.iq))
    assert len(lst) > nf
    with Engine("ble_wb40", max_samples=len(cap.iq), max_frames=max(nf, len(lst) - 1)) as e:
        e.run(cap.iq)
        with pytest.raises(_abi.SnrxError) as ei:
            e.ble_coded()
        assert ei.value.code == -6                              # SNRX_EOVERFLOW
    with Engine("ble_wb40", max_samples=len(cap.iq), max_frames=len(lst)) as e:
        e.run(cap.iq)
        assert e.ble_coded().tobytes() == lst.tobytes()


def legacy_capture(seconds=0.2, seed=9800):
    """Dense legacy traffic (1M advertising and data frames) on all 40 channels, 25 dB, no Coded packet."""
    rng = np.random.default_rng(seed)
    n_ch = int(round(seconds * chanplan.NB_RATE))
    n_ch -= n_ch % chanplan.BLE_WINDOW
    streams = {}
    for c in range(40):
        s, _ = synth.ble_baseband(n_ch, c, np.random.default_rng(seed + c), gap=(2000, 20000))
        streams[chanplan.ble_channel_bin(c)] = s
    x = synth.wideband_mix(streams)
    x = x + synth._awgn(len(x), np.random.default_rng(seed + 999), 4.0 * chanplan.WB_DECIM / 10 ** 2.5).astype(np.complex64)
    return x.astype(np.complex64)


def test_dense_legacy_capture_gives_no_coded_packet(Engine):
    """The false-alarm check of T: no Coded packet with a good CRC.  Uncoded 1M symbols are 4 samples long, so at a symbol
    boundary d(n) of legacy data has a deviation of 32, not the 16 of independent decisions: a few primaries with d <= T are
    expected there, and all of them fail the CRC.  Their count is printed."""
    x = legacy_capture()
    with Engine("ble_wb40", max_samples=len(x)) as e:
        frames = e.run(x)
        got = e.ble_coded()
        want = expected(e, len(x) // 24)
    assert_coded_equal(got, want, "legacy")
    assert len(frames) > 500
    prim = got[got["depth"] == 0]
    print(f"dense legacy capture: {len(frames)} records, {len(prim)} primaries with d <= T, "
          f"{int((prim['status'] == _abi.AUX_OK).sum())} decoded, {int(prim['crc_ok'].sum())} with a good CRC")
    assert not prim["crc_ok"].any() and not (got["depth"] > 0).any()


# S=8 recall of the Coded primaries the numpy chain model gives (tests/test_ble_coded.chain_recall, 40 packets, seed 7)
CPU_S8_RECALL = {4.0: 0.0, 6.0: 0.0, 7.0: 0.45, 8.0: 0.825, 9.0: 1.0, 10.0: 1.0}
# the engine at 4 dB, where it is not yet at 1.0: 51 of 60 measured (NVIDIA B200); pinned with a margin
ENGINE_S8_FLOOR = {4.0: 0.7}


@pytest.mark.parametrize("esn0", [4.0, 6.0, 8.0, 10.0])
def test_low_snr_recall_against_the_cpu_chain(Engine, esn0):
    """S=8 primaries at a low Es/N0 (synth's definition): the engine recovers at least what the CPU chain model recovers at
    the same Es/N0.  The model feeds white noise over the whole 4 MHz channel rate to the slicer; the engine's channel filter
    passes about a quarter of it, so the engine is expected to do better (DESIGN 4).  The measured recall is printed."""
    cap = synth.coded_adv_capture(seconds=0.3, seed=9750 + int(esn0), esn0_db=esn0, n_events=20, max_chain=0, s_values=(8,),
                                  phys=(0,))
    truth = [t for t in cap.meta["coded"] if t.depth == 0]
    with Engine("ble_wb40", max_samples=len(cap.iq)) as e:
        e.run(cap.iq)
        got = e.ble_coded()
    rec = recovered(got[got["depth"] == 0], truth) / len(truth)
    print(f"Es/N0 {esn0} dB: S=8 primaries recovered {rec:.3f} of {len(truth)} (CPU chain model: {CPU_S8_RECALL[esn0]:.3f}, "
          f"1 dB lower: {CPU_S8_RECALL.get(esn0 - 1, 0.0):.3f})")
    assert rec >= max(CPU_S8_RECALL[esn0], ENGINE_S8_FLOOR.get(esn0, 0.0))
