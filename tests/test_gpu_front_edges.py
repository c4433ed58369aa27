"""The front ends at their edges, stage by stage against their definitions: the quantiser that links the channel streams (S1)
to the quantised streams the frames are stated on (S2), the slicer bits, capture lengths that end anywhere inside a tile,
block or word, stride padding that is not zero, engines whose buffers hold an earlier, larger batch, and the chunked
staging of host input.  Every capture is small; the rules are in tests/quant_rule.py."""
import numpy as np
import pytest

from conftest import assert_frames_equal, ble_expected
from quant_rule import check_q8, quantize, slicer_words
from snout_b200 import _abi, chanplan, synth

pytestmark = pytest.mark.gpu

CHAN_TOL = 1e-4                # channelizer: max |err| / rms of the channel streams (as test_gpu_parity)
WB_MODES = ("ble_wb40", "zb_wb16", "mixed_wb56")
BLE_CH, ZB_CH = 17, 20         # narrow-band channels
HAS_BLE = ("ble_nb", "ble_wb40", "mixed_wb56")
HAS_ZB = ("zb_nb", "zb_wb16", "mixed_wb56")
KIND = {"ble_wb40": "ble", "zb_wb16": "zigbee", "mixed_wb56": "mixed"}


@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"

    def make(mode, **kw):
        kw.setdefault("max_frames", 1 << 13)
        if mode in ("ble_nb", "zb_nb"):
            kw.setdefault("channel", BLE_CH if mode == "ble_nb" else ZB_CH)
        return RxEngine(mode, **kw)
    return make


def _stages(e, mode):
    """Every stream a keep_streams engine holds for its last batch."""
    s = {}
    if mode in HAS_BLE:
        s["q8"] = e.debug_stage(_abi.STAGE_BLE_Q8)
        s["bits"] = e.debug_stage(_abi.STAGE_BLE_BITS)
    if mode in WB_MODES:
        s["y"] = e.debug_stage(_abi.STAGE_CHAN_CF32)
    if mode in HAS_ZB:
        s["f"] = e.debug_stage(_abi.STAGE_ZB_F)
        s["z"] = e.debug_stage(_abi.STAGE_ZB_DISC)
        s["nchips"] = e.debug_stage(_abi.STAGE_ZB_NCHIPS)
        s["chips"] = e.debug_stage(_abi.STAGE_ZB_CHIPS)
    return s


def _run(e, mode, x, **kw):
    fr = e.run(x, **kw)
    return fr, _stages(e, mode)


def _canon(fr):
    return fr[np.lexsort((fr["sample_index"], fr["window"], fr["channel"], fr["proto"], fr["capture_id"]))]


def _of_capture(st, k):
    """Streams of capture k of a batch (the chains of a batch are ordered (capture, channel, segment))."""
    out = {}
    for name, a in st.items():
        if name in ("nchips", "chips"):
            per = len(a) // (len(st["f"]))
            out[name] = a[k * per:(k + 1) * per]
        else:
            out[name] = a[k: k + 1]
    return out


def _assert_stages_equal(got, want, what):
    assert set(got) == set(want), what
    for name in want:
        if name == "chips":
            continue
        assert got[name].shape == want[name].shape, f"{what}: {name} shape {got[name].shape} vs {want[name].shape}"
        assert np.array_equal(got[name], want[name]), f"{what}: stage {name} differs"
    if "chips" in want:
        for k, nc in enumerate(want["nchips"]):
            assert np.array_equal(got["chips"][k, :nc], want["chips"][k, :nc]), f"{what}: soft chips of chain {k}"


def _zb_chips_check(st, k, c, n_ch, zo, seg, pre, what):
    n_seg = -(-len(zo) // seg)
    nchips, chips = st["nchips"], st["chips"]
    for j in range(n_seg):
        lo, hi = j * seg, min(len(zo), (j + 1) * seg)
        _, ck, _ = _oracle().zb_chain(zo, max(0, lo - pre), min(len(zo), hi + 16448), lo, hi, want_chips=True, hold=lo - 1024)
        chain = (k * n_ch + c) * n_seg + j
        assert nchips[chain] == len(ck), f"{what}: chain {chain} made {nchips[chain]} chips, expected {len(ck)}"
        assert np.array_equal(chips[chain, : len(ck)], ck), f"{what}: soft chips of chain {chain}"


def _oracle():
    import oracle
    return oracle


def _check_oracle(Engine, mode, x, fr, st, k=0, taps=384, seg=4096, pre=2048, scale=None, yd_ble=None, what=""):
    """Capture k of a batch (input x, cf32 [n]): every stream and the frames against the oracle.  yd_ble: the channelizer
    statement of x's BLE channels, when the caller has it."""
    o = _oracle()
    wide = mode in WB_MODES
    n_out = len(x) // 24 if wide else len(x)
    want = []
    if mode == "ble_nb":
        s = 128.0 if scale is None else scale
        q8 = o.ble_quantize(x, s)
        assert np.array_equal(st["q8"][k, 0], q8), f"{what}: q8"
        assert np.array_equal(st["bits"][k, 0], slicer_words(q8)), f"{what}: slicer bits"
        want.append(ble_expected(o, q8, BLE_CH))
    if mode in ("ble_wb40", "mixed_wb56"):
        y = st["y"][k]
        assert y.shape == (40, n_out), (what, y.shape)
        if yd_ble is None:
            yd_ble = o.pfb(x, _abi.pfb_prototype(_abi.MODE_BLE_WB40, taps), [chanplan.ble_channel_bin(c) for c in range(40)])
        rms = np.sqrt(np.mean(np.abs(yd_ble) ** 2))
        assert np.abs(y - yd_ble).max() <= CHAN_TOL * rms, f"{what}: BLE channel streams"
        q8 = st["q8"][k]
        check_q8(q8, y, yd_ble, 100.0 if scale is None else scale, what=what)
        assert np.array_equal(st["bits"][k], slicer_words(q8)), f"{what}: slicer bits"
        want += [ble_expected(o, q8[c], c) for c in range(40)]
    if mode == "zb_nb":
        fo = o.zb_quad_demod(x)
        assert np.array_equal(st["f"][k, 0], fo), f"{what}: discriminator"
        zo = o.zb_dc_remove(fo)
        assert np.array_equal(st["z"][k, 0], zo), f"{what}: DC removal"
        _zb_chips_check(st, k, 0, 1, zo, seg, pre, what)
        want.append(o.zb_receive(x, ZB_CH, segment=seg, prehalo=pre))
    if mode in ("zb_wb16", "mixed_wb56"):
        if mode == "zb_wb16":
            yz = st["y"][k]
            ydz = o.pfb(x, _abi.pfb_prototype(_abi.MODE_ZB_WB16, taps), [chanplan.zigbee_channel_bin(c) for c in range(11, 27)])
            assert np.abs(yz - ydz).max() <= CHAN_TOL * np.sqrt(np.mean(np.abs(ydz) ** 2)), f"{what}: 802.15.4 channel streams"
        else:                                  # the mixed engine keeps the BLE streams only: the 802.15.4 ones of a zb_wb16 engine
            with Engine("zb_wb16", max_samples=len(x), pfb_taps=taps, keep_streams=True, zb_segment=seg, zb_prehalo=pre) as ez:
                ez.run(x)
                yz = ez.debug_stage(_abi.STAGE_CHAN_CF32)[0]
        for c in range(16):
            fo = o.zb_quad_demod(yz[c])
            assert np.array_equal(st["f"][k, c], fo), f"{what}: discriminator of channel {11 + c}"
            zo = o.zb_dc_remove(fo)
            assert np.array_equal(st["z"][k, c], zo), f"{what}: DC removal of channel {11 + c}"
            _zb_chips_check(st, k, c, 16, zo, seg, pre, f"{what}, channel {11 + c}")
            want.append(o.zb_receive_z(zo, 11 + c, segment=seg, prehalo=pre))
    want = np.concatenate(want)
    want["capture_id"] = k
    got = fr[fr["capture_id"] == k]
    assert_frames_equal(_canon(got), _canon(want), what=f"{what}: frames")
    return len(want)


def _grid_captures(mode, n, seeds):
    """Captures on the int8 grid / 128 (so that their sc8 form is the same input) and the quantiser scale that reads them
    as the engine's default scale reads the unquantised capture (None: the mode's default)."""
    if mode == "ble_nb":
        return [synth.ble_capture(n=n, channel=BLE_CH, seed=s, esn0_db=28.0, gap=(100, 1500)).iq for s in seeds], None
    if mode == "zb_nb":
        xs = [synth.zigbee_capture(n=n, channel=ZB_CH, seed=s, esn0_db=20.0, gap=(300, 3000)).iq for s in seeds]
        peak = 1.0
    else:
        xs = [synth.wideband_capture(seconds=0.0042, kind=KIND[mode], seed=s, esn0_db=25.0, gap=(300, 2500)).iq[:n]
              for s in seeds]
        peak = max(float(np.abs(x.view(np.float32)).max()) for x in xs)
    q = [np.clip(np.rint(x.view(np.float32) * (100.0 / peak)), -128, 127) for x in xs]
    return [(v.astype(np.float32) / 128.0).view(np.complex64) for v in q], (128.0 * peak if mode in WB_MODES else None)


# ------------------------------------------------------------------------------------ 1. the quantiser
@pytest.mark.parametrize("taps", [384, 768])
def test_wideband_quantiser_against_definition(Engine, oracle_mod, taps):
    cap = synth.wideband_capture(seconds=0.0085, kind="ble", seed=4000, gap=(200, 2500))
    x = cap.iq[: len(cap.iq) - 24 * 40]
    with Engine("ble_wb40", max_samples=len(x), pfb_taps=taps, keep_streams=True) as e:
        e.run(x)
        q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0]
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
    yd = oracle_mod.pfb(x, _abi.pfb_prototype(_abi.MODE_BLE_WB40, taps), [chanplan.ble_channel_bin(c) for c in range(40)])
    excluded, bias = check_q8(q8, y, yd, 100.0, what=f"ble_wb40, {taps} taps")
    print(f"ble_wb40 {taps} taps: {excluded:.3%} of {q8.size} components within the margin of a step boundary, bias {bias:.1e}")


def test_mixed_quantiser_against_definition(Engine, oracle_mod):
    x = synth.wideband_capture(seconds=0.0085, kind="mixed", seed=5000, esn0_db=25.0, gap=(400, 5000)).iq
    with Engine("mixed_wb56", max_samples=len(x), keep_streams=True) as e:
        e.run(x)
        q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0]
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
    yd = oracle_mod.pfb(x, _abi.pfb_prototype(_abi.MODE_BLE_WB40, 384), [chanplan.ble_channel_bin(c) for c in range(40)])
    excluded, bias = check_q8(q8, y, yd, 100.0, what="mixed_wb56 BLE half")
    print(f"mixed_wb56: {excluded:.3%} of {q8.size} components within the margin of a step boundary, bias {bias:.1e}")


def test_wideband_quantiser_saturates_exactly(Engine, oracle_mod):
    """A scale at which more than 1 % of the components lie beyond each end of the int8 grid: they read -128 and 127."""
    cap = synth.wideband_capture(seconds=0.005, kind="ble", seed=4400, gap=(100, 800))
    x = cap.iq
    yd = oracle_mod.pfb(x, _abi.pfb_prototype(_abi.MODE_BLE_WB40, 384), [chanplan.ble_channel_bin(c) for c in range(40)])
    v = np.stack([yd.real, yd.imag], -1).astype(np.float64)
    s = float(np.float32(1.1 * max(128.5 / -np.quantile(v, 0.015), 127.5 / np.quantile(v, 0.985))))
    with Engine("ble_wb40", max_samples=len(x), keep_streams=True, quant_scale=s) as e:
        e.run(x)
        q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0].astype(np.int64)
        y = e.debug_stage(_abi.STAGE_CHAN_CF32)[0]
    lo, hi = v * s < -128.5, v * s > 127.5
    assert lo.mean() > 0.01 and hi.mean() > 0.01
    assert np.all(q8[lo] == -128) and np.all(q8[hi] == 127)
    assert q8.min() == -128 and q8.max() == 127
    check_q8(q8, y, yd, s, what=f"ble_wb40 at scale {s}")


def _edge_values(scale):
    k = np.arange(-130, 130)
    tiny = np.finfo(np.float32).tiny
    v = np.concatenate([(k + 0.5) / scale, np.nextafter(((k + 0.5) / scale).astype(np.float32), np.float32(np.inf)),
                        [0.0, -0.0, 1.0, -1.0, 127.49 / scale, 127.5 / scale, -128.5 / scale, -128.51 / scale, 1.5, -1.5, 7.0,
                         -7.0, 1e30, -1e30, tiny, -tiny, tiny / 8, -tiny / 8, 1.4e-45, -1.4e-45]])
    return v.astype(np.float32)


@pytest.mark.parametrize("scale", [128.0, 256.0, 100.0])
def test_narrowband_quantiser_edges(Engine, oracle_mod, scale):
    """Exact ties (k + 1/2) / S for k = -130 .. 129, +-0, values beyond full scale, subnormals: the engine's q8 is the
    oracle's, and the oracle's is clamp(rint(float32(x) * float32(S)))."""
    v = _edge_values(scale)
    rng = np.random.default_rng(int(scale))
    iq = np.stack([v, rng.permutation(v)], -1)
    iq = np.concatenate([iq, rng.uniform(-1.1, 1.1, (4096 + 3 - len(iq), 2)).astype(np.float32)])
    x = np.ascontiguousarray(iq).view(np.complex64).reshape(-1)
    want = oracle_mod.ble_quantize(x, scale)
    with np.errstate(over="ignore"):
        definition = quantize(np.rint(iq * np.float32(scale)))
    assert np.array_equal(want, definition.astype(np.int8))
    assert (want == -128).sum() > 10 and (want == 127).sum() > 10
    with Engine("ble_nb", max_samples=len(x), keep_streams=True, quant_scale=scale) as e:
        e.run(x)
        q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0, 0]
        bits = e.debug_stage(_abi.STAGE_BLE_BITS)[0, 0]
    assert np.array_equal(q8, want)
    assert np.array_equal(bits, slicer_words(want))


# ------------------------------------------------------------------------------------ 2. the slicer
@pytest.mark.parametrize("mode", ["ble_nb", "ble_wb40", "mixed_wb56"])
def test_slicer_bits_of_the_production_build(Engine, oracle_mod, mode):
    """Bit n = I[n] Q[n+1] - I[n+1] Q[n] > 0 on q8, last successor 0; lead words and words past the capture zero."""
    if mode == "ble_nb":
        x = synth.ble_capture(n=8192 * 3 + 1001, channel=BLE_CH, seed=31, esn0_db=28.0, gap=(100, 1500)).iq
        q8 = oracle_mod.ble_quantize(x, 128.0)[None]
    else:
        x = synth.wideband_capture(seconds=0.0045, kind=KIND[mode], seed=4600, esn0_db=25.0, gap=(300, 2500)).iq
        x = x[: len(x) - 24 * 13]
        with Engine(mode, max_samples=len(x), keep_streams=True) as e:
            e.run(x)
            q8 = e.debug_stage(_abi.STAGE_BLE_Q8)[0]
            kept = e.debug_stage(_abi.STAGE_BLE_BITS)[0]
        assert np.array_equal(kept, slicer_words(q8))
    with Engine(mode, max_samples=len(x)) as e:
        fr = e.run(x)
        bits = e.debug_stage(_abi.STAGE_BLE_BITS)[0]
    want = slicer_words(q8)
    assert bits.shape == want.shape
    for c in range(len(want)):
        assert np.array_equal(bits[c], want[c]), f"{mode}: slicer words of stream {c}"
    assert len(fr) > 3


# ------------------------------------------------------------------------------------ 3. lengths
def _sweep(Engine, mode, x_full, lengths, taps=384, **cfg):
    """Run every prefix x_full[:n] (n channel samples) on a fresh engine; check it stage by stage against the oracle.  Every
    length given is one the engine supports: a refusal is a failure."""
    wide = mode in WB_MODES
    yd = None
    if mode in ("ble_wb40", "mixed_wb56"):
        n_max = max(lengths)
        yd = _oracle().pfb(x_full[: n_max * 24], _abi.pfb_prototype(_abi.MODE_BLE_WB40, taps),
                           [chanplan.ble_channel_bin(c) for c in range(40)])
    errors, frames = [], 0
    for n in lengths:
        x = x_full[: n * 24 if wide else n].copy()
        with Engine(mode, max_samples=len(x), pfb_taps=taps, keep_streams=True, **cfg) as e:
            try:
                fr = e.run(x)
            except _abi.SnrxError as err:
                errors.append(f"length {n}: refused ({err})")
                continue
            st = _stages(e, mode)
        try:
            frames += _check_oracle(Engine, mode, x, fr, st, taps=taps, yd_ble=None if yd is None else yd[:, :n],
                                    seg=cfg.get("zb_segment", 4096), pre=cfg.get("zb_prehalo", 2048), what=f"{mode} length {n}")
        except AssertionError as err:
            errors.append(str(err).splitlines()[0])
    assert not errors, "\n".join(errors)
    return frames


def test_ble_nb_lengths(Engine):
    cap = synth.ble_capture(n=8192 * 3, channel=BLE_CH, seed=41, esn0_db=28.0, gap=(60, 700))
    ends = [t.start + 4 * (8 + 32 + 8 * len(t.data)) + 16 for t in cap.truth]
    n_end = max(v for v in ends if v < len(cap.iq) - 8) + 3          # three samples past the end of the last whole burst
    lengths = [1, 2, 31, 32, 33, 127, 128, 129, 159, 160, 161, 8191, 8192, 8193, n_end, 8192 * 3]
    assert _sweep(Engine, "ble_nb", cap.iq, lengths) > 10


def test_zb_nb_lengths(Engine):
    cap = synth.zigbee_capture(n=1_000_003, channel=ZB_CH, seed=43, esn0_db=18.0, gap=(300, 5000))
    lengths = [1, 2, 3, 5, 6, 7, 2047, 2049, 2050, 2051, 4095, 4097, 4098, 4099, 6145, 8190, 8193, 12_291, 1_000_003]
    assert _sweep(Engine, "zb_nb", cap.iq, lengths) > 20


WB_LENGTHS = [1, 2, 15, 30, 31, 32, 33, 62, 63, 127, 128, 129, 8191, 8192, 8193, 8214]


@pytest.mark.parametrize("taps", [384, 768])
@pytest.mark.parametrize("mode", WB_MODES)
def test_wideband_lengths(Engine, mode, taps):
    """n_out shorter than the tap history, one tile, n_out = 0, 1, 30 (mod 31), across a window; a capture that is not a
    whole number of channel samples is refused."""
    x = synth.wideband_capture(seconds=0.0045, kind=KIND[mode], seed=4700, esn0_db=25.0, gap=(100, 1500)).iq
    assert len(x) >= 24 * max(WB_LENGTHS)
    frames = _sweep(Engine, mode, x, WB_LENGTHS, taps=taps)
    assert frames > (20 if mode != "zb_wb16" else 0)
    with Engine(mode, max_samples=24 * 200, pfb_taps=taps) as e:
        for n in (1, 23, 25, 24 * 100 + 7):
            with pytest.raises(_abi.SnrxError):
                e.run(x[:n].copy())


# ------------------------------------------------------------------------------------ 4. stride padding
@pytest.mark.parametrize("mode", ["ble_nb", "zb_nb", "ble_wb40", "zb_wb16", "mixed_wb56"])
def test_batch_with_loud_stride_padding(Engine, mode):
    """Three captures at stride n + 2k whose padding holds loud values: device cf32, device and host sc8, host cf32.  Every
    stream and frame of each capture equals its single run, and each single run equals the oracle stage by stage."""
    import torch
    wide = mode in WB_MODES
    n = 24 * (8192 + 777) if wide else 8192 * 4 + 1234
    k = 50
    caps, scale = _grid_captures(mode, n, [4800 + 17 * i for i in range(3)])
    kw = dict(max_samples=n, keep_streams=True, **({"quant_scale": scale} if scale else {}))
    singles, frames_single, n_frames = [], [], 0
    for i, c in enumerate(caps):
        with Engine(mode, **kw) as e:
            fr, st = _run(e, mode, c)
        n_frames += _check_oracle(Engine, mode, c, fr, st, scale=scale, what=f"{mode} capture {i} alone")
        fr["capture_id"] = i
        frames_single.append(fr)
        singles.append(st)
    assert n_frames > 3
    want_frames = _canon(np.concatenate(frames_single))
    xp = np.full((3, n + 2 * k), 0.9 + 0.9j, np.complex64)
    xp[:, :n] = np.stack(caps)
    q = np.rint(np.stack(caps).view(np.float32).reshape(3, n, 2) * 128.0).astype(np.int8)
    qp = np.full((3, n + 2 * k, 2), 127, np.int8)
    qp[:, :n] = q
    with Engine(mode, max_captures=3, **kw) as e:
        for name, inp in (("device cf32", torch.from_numpy(xp).cuda()), ("device sc8", torch.from_numpy(qp).cuda()),
                          ("host sc8", qp), ("host cf32", xp)):
            fr, st = _run(e, mode, inp, n_samples=n, stride=n + 2 * k)
            assert_frames_equal(_canon(fr), want_frames, what=f"{mode}, {name} batch: frames")
            for i in range(3):
                _assert_stages_equal(_of_capture(st, i), singles[i], f"{mode}, {name} batch, capture {i}")


# ------------------------------------------------------------------------------------ 5. dirty engines
def _loud(mode, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.uniform(-1.0, 1.0, (n, 2)).astype(np.float32)).view(np.complex64).reshape(-1)


def _short_batch(mode, channel=None):
    if mode == "ble_nb":
        n = 8192 + 4097
        caps = [synth.ble_capture(n=n, channel=channel or BLE_CH, seed=60 + i, esn0_db=28.0, gap=(100, 1200)).iq for i in range(2)]
    elif mode == "zb_nb":
        n = 40_001
        caps = [synth.zigbee_capture(n=n, channel=channel or ZB_CH, seed=61 + i, esn0_db=20.0, gap=(300, 2000)).iq for i in range(2)]
    else:
        n = 24 * 10_209
        caps = [synth.wideband_capture(seconds=0.0042, kind=KIND[mode], seed=4800 + i, esn0_db=25.0, gap=(100, 900)).iq[:n]
                for i in range(2)]
    stride = n + (n & 1) + 6
    xp = np.full((2, stride), -0.95 + 0.7j, np.complex64)
    xp[:, :n] = np.stack(caps)
    return xp, n, stride


@pytest.mark.parametrize("mode", ["ble_nb", "zb_nb", "ble_wb40", "zb_wb16", "mixed_wb56"])
def test_dirty_engine_equals_fresh_engine(Engine, mode):
    """Both lanes of an engine run long, loud batches (one at max_captures), then a short ragged batch from host and from
    device memory: every stream and frame equals a fresh engine's.  Narrow band: again after set_channel."""
    import torch
    wide = mode in WB_MODES
    big = 24 * 12_000 if wide else 150_000
    cfg = dict(max_samples=big, max_captures=2, keep_streams=True)
    checks = [(None, None)]
    if mode == "ble_nb":
        checks.append((5, 5))
    elif mode == "zb_nb":
        checks.append((25, 25))
    with Engine(mode, **cfg) as e:
        e.run(_loud(mode, big, 1))
        e.run(_loud(mode, big, 2))
        e.run(np.stack([_loud(mode, big, 3), _loud(mode, big, 4)]))
        for set_to, ch in checks:
            if set_to is not None:
                e.set_channel(set_to)
            xp, n, stride = _short_batch(mode, ch)
            with Engine(mode, **cfg, **({"channel": ch} if ch else {})) as f:
                want_fr, want_st = _run(f, mode, xp, n_samples=n, stride=stride)
            assert len(want_fr) > (2 if mode in HAS_BLE else 0), (mode, ch)
            for name, inp in (("host", xp), ("device", torch.from_numpy(xp).cuda())):
                fr, st = _run(e, mode, inp, n_samples=n, stride=stride)
                what = f"{mode}, channel {ch}, {name} input after loud batches"
                assert_frames_equal(fr, want_fr, what=what)
                _assert_stages_equal(st, want_st, what)
            e.run(_loud(mode, big, 5))                       # dirty again before the next check


# ------------------------------------------------------------------------------------ 6. pipelined host staging
@pytest.mark.parametrize("taps", [384, 768])
def test_pipelined_host_staging_equals_device_input(Engine, taps):
    """A single ble_wb40 capture from host memory is staged 4 Mi (cf32) / 8 Mi (sc8) samples at a time, with the channelizer
    launched on the tiles whose input has arrived: the slicer bits equal those of the same capture from device memory,
    when the last chunk is short and when it holds less than one tile."""
    import torch
    base = synth.wideband_capture(seconds=0.02, kind="ble", seed=4900, gap=(200, 3000)).iq
    peak = float(np.abs(base.view(np.float32)).max())
    up = lambda v: -(-v // 24) * 24                                  # noqa: E731
    for fmt, chunk in (("cf32", 4 << 20), ("sc8", 8 << 20)):
        for n in (up(2 * chunk + 30_000), up(chunk + 1)):
            x = np.resize(base, n)
            if fmt == "sc8":
                x = np.clip(np.rint(x.view(np.float32).reshape(-1, 2) * (100.0 / peak)), -128, 127).astype(np.int8)
            with Engine("ble_wb40", max_samples=n, pfb_taps=taps, max_frames=1 << 16) as e:
                a = e.run(x)
                bits_host = e.debug_stage(_abi.STAGE_BLE_BITS)
                b = e.run(torch.from_numpy(x).cuda())
                bits_dev = e.debug_stage(_abi.STAGE_BLE_BITS)
            what = f"{fmt}, {taps} taps, n = {n} (last chunk {n % chunk} samples)"
            assert len(a) > 100, what
            assert np.array_equal(bits_host, bits_dev), what
            assert_frames_equal(a, b, what=what)
