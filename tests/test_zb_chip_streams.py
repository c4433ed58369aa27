"""The 802.15.4 back end on constructed chip streams (tests/zb_chips.py), on the CPU: every case hits the edge it is built
for on the oracle, the host build of the kernels' chain code (tests/emu) equals the oracle on it, the windowed sink equals
the chip-by-chip sink on its chips, a chain's frame slots hold the densest run that decodes, and k_zb_rx's tracker pacing
(catch-up and pause windows) is restated over the oracle's chip positions."""
import ctypes
import functools

import numpy as np
import pytest

import zb_chips as Z
from conftest import assert_frames_equal
from snout_b200 import synth

P = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731


@functools.lru_cache(maxsize=None)
def _cases():
    return {c.name: c for c in Z.cases()}


NAMES = [c.name for c in Z.cases()]


@pytest.mark.parametrize("name", NAMES)
def test_case_hits_its_edge_on_the_oracle(oracle_mod, name):
    case = _cases()[name]
    case.check(oracle_mod, case, Z.oracle_frames(oracle_mod, case))


def _emu_chains(emu, oracle_mod, z, case):
    n = len(z)
    out = np.zeros(4096, dtype=oracle_mod.FRAME_DTYPE)
    nseg = -(-n // case.segment)
    nch = np.zeros(nseg, np.int64)
    k = emu.emu_zb_chains(P(z), n, 0, n, case.segment, case.prehalo, ctypes.c_uint32(0), case.threshold, Z.CHANNEL, P(out),
                          len(out), P(nch))
    return k, out[:max(k, 0)].copy(), nch


@pytest.mark.parametrize("name", NAMES)
def test_emu_chains_equal_the_oracle(oracle_mod, emu, name):
    """zb_run_chain + zb_filter_chain (the per-thread code of k_zb_rx and k_zb_span_filter) with the chain's slot count:
    the oracle's records field for field, and every chain stops at the oracle's chip.  A chain that finds more records
    than its slots is reported, not clamped."""
    case = _cases()[name]
    for i, x in enumerate(case.captures):
        z = oracle_mod.zb_dc_remove(oracle_mod.zb_quad_demod(x))
        k, got, nch = _emu_chains(emu, oracle_mod, z, case)
        assert k >= 0, f"{name}: chain {-k - 1} found more records than its {emu.emu_zb_slots_per_chain(case.segment)} slots"
        want = oracle_mod.zb_receive(x, Z.CHANNEL, threshold=case.threshold, segment=case.segment, prehalo=case.prehalo)
        assert_frames_equal(got, want, what=f"{name} capture {i}")
        for c, (lo, hi, begin, end) in enumerate(Z.chain_geometry(len(z), case.segment, case.prehalo)):
            _, ck, _ = oracle_mod.zb_chain(z, begin, end, lo, hi, threshold=case.threshold, want_chips=True, hold=lo - Z.SINK_LEAD)
            assert nch[c] == len(ck), (name, c)


def _port_sink(oracle_mod, chips, thr):
    lib = oracle_mod._lib("port")
    st = ctypes.create_string_buffer(lib.zb_oracle_sink_size())
    lib.zb_sink_init(st, thr)
    lib.zb_sink_psdu.restype = ctypes.POINTER(ctypes.c_uint8)
    out = []
    for i, c in enumerate(chips):
        if lib.zb_sink_push(st, int(c), ctypes.c_int64(i), ctypes.c_int64(i)):
            out.append((i, bytes(lib.zb_sink_psdu(st)[:lib.zb_sink_len(st)])))
    return out


def _window_sink(emu, chips, thr):
    hard = np.ascontiguousarray(chips, np.uint8)
    cap = 4096
    lens, by, endc = np.zeros(cap, np.int32), np.zeros((cap, 128), np.uint8), np.zeros(cap, np.int64)
    k = emu.emu_zb_sink_chips(P(hard), ctypes.c_int64(len(hard)), thr, P(lens), P(by), P(endc), cap)
    return [(int(endc[i]), bytes(by[i, :lens[i]])) for i in range(min(k, cap))]


@pytest.mark.parametrize("name", [n for n in NAMES if _cases()[n].chips])
def test_windowed_sink_equals_the_port_sink_on_constructed_chips(oracle_mod, emu, name):
    """zb_sink_window (32 chips at a time, resets at any offset of a window) against zb_sink_push, chip by chip, on the
    constructed chips -- and, where the chips are decided as constructed, the frames the receive chain reports are the
    port sink's."""
    case = _cases()[name]
    for chips in case.chips:
        want = _port_sink(oracle_mod, chips, case.threshold)
        assert _window_sink(emu, chips, case.threshold) == want
        if case.eps == 0.0 and not name.startswith("dense"):
            got = Z.oracle_frames(oracle_mod, case)
            assert [bytes(f["bytes"][:f["len"]]) for f in got] == [b for _, b in want]


def test_resets_at_every_window_offset(oracle_mod):
    """The dense run at threshold 12 publishes (and resets the register) 192 + 11 chips after each sync: the publishing
    chips fall on every offset 0..31 of the chain's 32-chip windows."""
    case = _cases()["dense_thr12"]
    z = oracle_mod.zb_dc_remove(oracle_mod.zb_quad_demod(case.iq))
    frames, ck, pos = oracle_mod.zb_chain(z, 0, len(z), 0, 65536, threshold=12, want_chips=True, hold=-Z.SINK_LEAD)
    sync = np.searchsorted(pos, frames["sample_index"])
    assert np.array_equal(pos[sync], frames["sample_index"]) and len(frames) == 48
    offsets = set(((sync + 128) % 32).tolist())
    assert offsets == set(range(32)), sorted(offsets)


def test_shard_edge_captures_sync_on_the_body_edges(oracle_mod):
    """The shard case of the GPU file: every capture's one frame syncs exactly on its edge of the shard body, and the
    shard's pre halo is the one the stream planner gives a Zigbee engine."""
    from snout_b200 import stream
    assert stream.shard_geometry(0, 1)[1] == Z.SHARD_PRE
    xs, targets, shard, lo = Z.shard_edge_captures()
    for x, t in zip(xs, targets):
        f = oracle_mod.zb_receive(x, Z.CHANNEL)
        assert list(f["sample_index"]) == [t] and f["crc_ok"].all() and f["window"][0] == t // Z.SEGMENT


def test_slot_count_holds_the_densest_decoding_run(oracle_mod, emu):
    """zb_slots_per_chain is the bound (S - 1) // 193 + 1 for a body of S samples: consecutive records of a chain sync at
    least 193 chips apart (PHR, one byte, one chip to re-lock, 7, 10) and every chip advances the clock recovery by at least
    one sample; that argument does not rest on any constructed stream.  What is checked against it: for thresholds 1..31,
    the densest plain run of len-0 frames (the k-chip tail of symbol 0 after each reset, k searched on the windowed sink)
    decodes up to threshold 12 and stays within the spacing; the former count, segment / 448 + 2, does not hold what the
    oracle decodes at 16384 and 65536.  Denser streams of other shapes at higher thresholds are not searched."""
    for seg in (2048, 4096, 8192, 16384, 32768, 65536):
        assert emu.emu_zb_slots_per_chain(seg) == Z.slots_bound(seg) == (seg - 1) // 193 + 1
    assert emu.emu_zb_slots_per_chain(4096) == 22
    densest = {}
    for thr in range(1, 32):
        for k in range(Z.relock_k(thr), 33):
            run = Z.dense_run(thr, 12, k)
            got = _window_sink(emu, run, thr)
            if len(got) == 12:
                spacing = np.diff([e for e, _ in got])
                assert (spacing == 192 + k).all() and 192 + k >= Z.MIN_SYNC_CHIPS
                densest[thr] = 192 + k
                break
    # the plain run decodes up to threshold 12; from 13 on the SFD's 7 is within thr of symbol 0 and reads as preamble
    assert sorted(densest) == list(range(1, 13)), densest
    assert densest[10] == 206 and densest[12] == 203 and min(densest.values()) >= Z.MIN_SYNC_CHIPS
    for name in ("dense_thr10_seg16384", "dense_thr10_seg65536", "dense_batch3"):
        case = _cases()[name]
        f = Z.oracle_frames(oracle_mod, case)
        per = np.unique(f["capture_id"].astype(np.int64) << 32 | f["window"], return_counts=True)[1]
        assert case.segment // 448 + 2 < per.max() <= emu.emu_zb_slots_per_chain(case.segment), (name, per.max())


def test_tracker_pacing_reaches_both_clamps_only_under_drift(oracle_mod, emu):
    """k_zb_rx's lead schedule (zb_chips.lead_schedule, with kZbLead / kZbLeadMin / kZbLeadMax as built) over the oracle's
    chip positions.  Chip-rate offsets of 1e-3 and 3e-3 make about a third of the windows catch up and a third pause, and
    every read keeps at least the 8 samples it needs, also in paused windows, and at most the 128 of the ring.  Natural
    traffic and white noise never leave the clamps: that is why the drift cases exist.  The worst case of a paused window
    is not reached by any input here; it is derived from the taps: at most 1 + 31 (2.0004 + 0.03 max|out|) samples of
    advance before the last read, max|out| <= max sum|taps| * 2 pi."""
    lead = np.zeros(3, np.int32)
    emu.emu_zb_lead_params(P(lead))
    lead = tuple(int(v) for v in lead)
    taps = np.zeros((129, 8), np.float32)
    emu.emu_zb_mmse_taps(P(taps))
    gain = float(np.abs(taps.astype(np.float64)).sum(axis=1).max())
    assert 1.5 < gain <= 1.60
    worst = 1 + 31 * (2.0004 + 0.03 * gain * 2 * np.pi)
    assert lead[2] + 1 - worst >= 8, (lead, worst)                 # a paused window's last read stays behind conv
    assert lead[1] - 32 - 8 >= 0, lead                            # an enabled window: 32 steps of 3 eat at most 32 of it
    assert lead[2] + 32 + 8 <= 128, lead                          # the ring
    for name in [n for n in NAMES if n.startswith("drift")]:
        s = Z.lead_schedule(oracle_mod, _cases()[name], lead)
        assert s["catch_up"] > s["windows"] // 5 and s["pause"] > s["windows"] // 5, (name, s)
        assert 8 <= s["min_read_lead"] and 8 <= s["min_paused_lead"] and s["max_read_lead"] <= 128, (name, s)
    rng = np.random.default_rng(3)
    noise = (rng.standard_normal(600_000) + 1j * rng.standard_normal(600_000)).astype(np.complex64)
    natural = [synth.zigbee_capture(n=600_000, channel=11, seed=s, esn0_db=15.0).iq for s in (2001, 2002, 77)] + [noise]
    for i, x in enumerate(natural):
        case = Z.Case(f"natural{i}", x, None, "")
        s = Z.lead_schedule(oracle_mod, case, lead)
        assert s["catch_up"] == 0 and s["pause"] == 0 and s["windows"] > 10_000, (i, s)
