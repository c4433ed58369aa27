"""BLE 5 extended advertising (snrx_ble_aux): the contract's restatement (oracle/aux_oracle.py) on constructed multi-channel
bit streams, end to end through the channelizer's CPU statement, and the host side (parsing, chain reassembly, pcap, CLI).
No GPU."""
import io
import struct

import numpy as np
import pytest

from ble_bits import ADV_AA, aa_bits, lsb_bits, pack_words
from fake_engine import RecordingEngine
from oracle import aux_oracle as ao
from snout_b200 import _abi, btle_cli, chanplan, formats, messages, synth

N_CH = 40


# ------------------------------------------------------------------------------------------------ construction
def plant_stride(b: np.ndarray, s: int, symbols, sps: int) -> None:
    """b[s + k sps] = symbols[k]; those outside the stream are dropped (ble_bits.plant at any stride)."""
    symbols = np.asarray(symbols, dtype=np.uint8)
    pos = s + sps * np.arange(len(symbols))
    ok = (pos >= 0) & (pos < len(b))
    b[pos[ok]] = symbols[ok]


def aux_symbols(channel: int, pdu: bytes, crc_ok: bool = True) -> np.ndarray:
    """AA | whiten(pdu | CRC-24) as symbols, from synth's whitening / CRC definitions."""
    crc = bytearray(synth.ble_crc24(pdu))
    if not crc_ok:
        crc[2] ^= 0x01
    body = np.frombuffer(bytes(pdu) + bytes(crc), np.uint8) ^ synth.ble_whitening(channel, len(pdu) + 3)
    return np.concatenate([aa_bits(ADV_AA), lsb_bits(body.tobytes())])


def primary_record(s: int, ptr: bytes, channel: int = 37, capture_id: int = 0, adi: int | None = 0x1234) -> np.void:
    pdu = synth.ext_pdu(synth.ext_header(0, None, 0, adi, ptr))
    data = pdu + synth.ble_crc24(pdu)
    f = np.zeros(1, _abi.FRAME_DTYPE)[0]
    f["sample_index"], f["capture_id"], f["channel"], f["proto"], f["crc_ok"] = s, capture_id, channel, 3, 1
    f["len"], f["access_addr"] = len(data), ADV_AA
    f["bytes"][: len(data)] = np.frombuffer(data, np.uint8)
    return f


class Batch:
    """Bit streams of every channel of one capture (random fill) and the records pointing into them."""

    class _Chans(dict):
        def __init__(self, n, rng):
            super().__init__()
            self.n, self.rng = n, rng

        def __missing__(self, c):
            self[c] = self.rng.integers(0, 2, self.n, dtype=np.uint8)     # a channel's fill is drawn when it is first used
            return self[c]

    def __init__(self, n: int, seed: int = 0):
        self.n = n
        self.b = Batch._Chans(n, np.random.default_rng(abs(seed)))
        self.frames = []

    def words(self):
        nw = 4 + (self.n + 31) // 32 + 64
        w = np.zeros((1, N_CH, nw), np.uint32)
        for c, b in self.b.items():
            w[0, c] = pack_words(b, n_words=nw)
        return w

    def run(self, **kw):
        fr = np.array(self.frames, dtype=_abi.FRAME_DTYPE) if self.frames else np.zeros(0, _abi.FRAME_DTYPE)
        return ao.aux_list(self.words(), fr, self.n, **kw)


def aux_pdu(rng, adv_len: int, ptr: bytes | None = None) -> bytes:
    hdr = synth.ext_header(0, bytes(rng.integers(0, 256, 6, dtype=np.uint8)), 0, int(rng.integers(0, 1 << 16)), ptr, -7)
    return synth.ext_pdu(hdr, bytes(rng.integers(0, 256, adv_len - len(hdr), dtype=np.uint8)))


def check_decoded(r, channel: int, pdu: bytes, crc_ok: bool = True):
    want = pdu + synth.ble_crc24(pdu)
    assert r["status"] == ao.OK and r["channel"] == channel
    assert r["len"] == len(want) and bytes(r["bytes"][: len(want)]) == (want if crc_ok else bytes(r["bytes"][: len(want)]))
    assert not r["bytes"][len(want):].any()
    assert bool(r["crc_ok"]) == crc_ok


# ------------------------------------------------------------------------------------------------ the definitions
def test_lfsr_and_crc_definitions_agree_with_synth():
    for ch in (0, 5, 36, 37, 39):
        assert np.array_equal(ao.whitening(ch, 260), synth.ble_whitening(ch, 260))
    rng = np.random.default_rng(1)
    for n in (0, 1, 2, 40, 257):
        d = bytes(rng.integers(0, 256, n, dtype=np.uint8))
        c = synth.ble_crc24(d)
        assert ao.crc24_ok(d, c) and not ao.crc24_ok(d, bytes([c[0] ^ 1, c[1], c[2]]))


def test_aux_ptr_fields_and_window_arithmetic():
    p = synth.aux_ptr_bytes(21, 1, 300, 8191, 1)
    pdu = synth.ext_pdu(synth.ext_header(0, b"\1" * 6, 0, 7, p))
    assert ao.parse_aux_ptr(pdu, pdu[1]) == (21, 1, 300, 8191, 1)
    assert ao.window(30, 0, 1) == (-8, 120 + 8 + 1)                  # ceil(4 * 30 * 1.00005) = 121
    assert ao.window(300, 8191, 0) == ((4 * 2457300 * 999500) // 10**6 - 8, -((-4 * 2457600 * 1000500) // 10**6) + 8)
    # header too short for the fields in front of the AuxPtr, or no AuxPtr flag: not a pointer
    short = bytes([7, 8, 5, 0x19]) + b"\1" * 6
    assert ao.parse_aux_ptr(short, short[1]) is None
    assert ao.parse_aux_ptr(synth.ext_pdu(synth.ext_header(0, None, 0, 7, None)), 4) is None


# ------------------------------------------------------------------------------------------------ window edges
@pytest.mark.parametrize("ca", [0, 1])
@pytest.mark.parametrize("units,offset", [(30, 0), (30, 8191), (300, 0), (300, 8191), (30, 517)])
def test_window_edges(ca, units, offset):
    """AA exactly at win_lo and win_hi is found; one sample outside either is not."""
    rng = np.random.default_rng(units + offset + ca)
    lo, hi = ao.window(units, offset, ca)
    s = 300
    n = s + hi + 2000
    for where, found in ((lo, True), (hi, True), (lo - 1, False), (hi + 1, False)):
        bt = Batch(n, seed=offset + where)
        pdu = aux_pdu(rng, 20)
        bt.b[9] &= 0                                                  # nothing else that could match
        plant_stride(bt.b[9], s + where, aux_symbols(9, pdu), 4)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(9, ca, units, offset, 0)))
        (r,) = bt.run()
        assert (r["win_lo"], r["win_hi"]) == (s + lo, s + hi)
        if found:
            check_decoded(r, 9, pdu)
            assert r["sample_index"] == s + where and r["phase"] == (s + where) % 4
        else:
            assert r["status"] == ao.NOT_FOUND and r["sample_index"] == -1


@pytest.mark.parametrize("phase", [0, 1])
def test_2m_both_phases_and_earliest_match(phase):
    rng = np.random.default_rng(phase)
    bt = Batch(6000, seed=phase)
    s = 500
    lo, hi = ao.window(30, 20, 1)
    a, b_ = s + lo + 10 + phase, s + lo + 41 + phase          # two packets in the window: the earliest wins
    p1, p2 = aux_pdu(rng, 30), aux_pdu(rng, 40)
    plant_stride(bt.b[3], b_, aux_symbols(3, p2), 2)
    plant_stride(bt.b[3], a, aux_symbols(3, p1)[:32 + 16], 2)  # ... even if it is only an AA and a header
    plant_stride(bt.b[3], a, aux_symbols(3, p1), 2)
    bt.frames.append(primary_record(s, synth.aux_ptr_bytes(3, 1, 30, 20, 1)))
    (r,) = bt.run()
    check_decoded(r, 3, p1)
    assert r["sample_index"] == a and r["phase"] == a % 2 and r["phy"] == ao.PHY_2M


def test_every_length_and_crc_errors():
    """len 0..255 at both PHYs; every fifth packet with a wrong CRC."""
    rng = np.random.default_rng(7)
    bt = Batch(2_300_000, seed=7)
    s, want = 100, []
    for ln in range(256):
        sps = 4 if ln % 2 == 0 else 2
        pdu = synth.ext_pdu(b"", bytes(rng.integers(0, 256, ln, dtype=np.uint8))) if ln < 2 else aux_pdu(rng, max(ln, 12))[:2 + ln]
        pdu = bytes([pdu[0], ln]) + pdu[2:2 + ln]
        ok = ln % 5 != 3
        off = 3
        lo, _ = ao.window(30, off, 0)
        plant_stride(bt.b[11], s + lo + 8, aux_symbols(11, pdu, ok), sps)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(11, 0, 30, off, sps == 2)))
        want.append((pdu, ok))
        s += lo + 8 + sps * (40 + 8 * (ln + 5)) + 50
    got = bt.run()
    assert len(got) == 256
    for r, (pdu, ok) in zip(got, want):
        check_decoded(r, 11, pdu, ok)


def test_buffer_end_truncated_and_outside():
    rng = np.random.default_rng(3)
    pdu = aux_pdu(rng, 100)
    nbits = 32 + 8 * (len(pdu) + 3)
    for sps in (4, 2):
        lo, hi = ao.window(30, 2, 1)
        s = 200
        at = s + hi - 10                                           # late in the window: the header can be cut too
        end = at + (nbits - 1) * sps                               # last decision of the packet
        for n, status in ((end + 2, ao.OK), (end + 1, ao.TRUNCATED), (at + 47 * sps + 2, ao.TRUNCATED),
                          (at + 47 * sps + 1, ao.TRUNCATED)):
            bt = Batch(n, seed=n)
            plant_stride(bt.b[30], at, aux_symbols(30, pdu), sps)
            bt.frames.append(primary_record(s, synth.aux_ptr_bytes(30, 1, 30, 2, sps == 2)))
            (r,) = bt.run()
            assert r["status"] == status, (sps, n)
            if status == ao.TRUNCATED:
                assert r["sample_index"] == at and r["len"] == 0
        # the window plus the AA span must lie on usable decisions
        bt = Batch(s + hi + 31 * sps + 1, seed=1)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(30, 1, 30, 2, sps == 2)))
        assert bt.run()[0]["status"] == ao.OUTSIDE
        bt = Batch(s + hi + 31 * sps + 2, seed=1)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(30, 1, 30, 2, sps == 2)))
        assert bt.run()[0]["status"] != ao.OUTSIDE
    bt = Batch(5000)
    bt.frames.append(primary_record(5, synth.aux_ptr_bytes(30, 1, 30, 0, 0)))       # win_lo = -3 < 0
    assert bt.run()[0]["status"] == ao.OUTSIDE


def test_statuses_that_are_not_searched_and_sources():
    bt = Batch(5000)
    bt.frames.append(primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 2)))        # Coded
    bt.frames.append(primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 3)))        # reserved PHY
    bt.frames.append(primary_record(100, synth.aux_ptr_bytes(37, 0, 30, 3, 0)))       # channel index > 36
    f = primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 0)); f["crc_ok"] = 0; bt.frames.append(f)
    f = primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 0), channel=12); bt.frames.append(f)
    f = primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 0)); f["access_addr"] = 0x12345678; bt.frames.append(f)
    f = primary_record(100, synth.aux_ptr_bytes(5, 0, 30, 3, 0)); f["proto"] = 2; bt.frames.append(f)
    got = bt.run()
    assert list(got["status"]) == [ao.UNSUPPORTED_PHY, ao.UNSUPPORTED_PHY, ao.BAD_CHANNEL]
    assert list(got["parent"]) == [0, 1, 2] and list(got["first"]) == [0, 1, 2]


def _chain(bt, rng, s0: int, channels, phys, loop_last: bool = False):
    """A chain of len(channels) aux packets, each pointing at the next (the last points nowhere, or at itself)."""
    starts, t = [], s0 + 2000
    pdus = []
    for k in range(len(channels)):
        starts.append(t)
        t += 3000
    for k, (ch, phy) in enumerate(zip(channels, phys)):
        if k + 1 < len(channels):
            ptr = synth.aux_ptr_bytes(channels[k + 1], 1, 30, (starts[k + 1] - starts[k]) // 4 // 30, phys[k + 1])
        elif loop_last:
            ptr = synth.aux_ptr_bytes(ch, 1, 30, 0, phy)
        else:
            ptr = None
        pdu = aux_pdu(rng, 40, ptr)
        plant_stride(bt.b[ch], starts[k], aux_symbols(ch, pdu), 2 if phy else 4)
        pdus.append(pdu)
    ptr0 = synth.aux_ptr_bytes(channels[0], 1, 30, (starts[0] - s0) // 4 // 30, phys[0])
    return starts, pdus, ptr0


@pytest.mark.parametrize("links", [1, 2, 5, 15, 16, 17])
def test_chains_and_depth_limit(links):
    rng = np.random.default_rng(links)
    bt = Batch(2000 + 3000 * (links + 2), seed=links)
    chans = [int(c) for c in rng.integers(0, 37, links)]
    phys = [int(p) for p in rng.integers(0, 2, links)]
    starts, pdus, ptr0 = _chain(bt, rng, 100, chans, phys)
    bt.frames.append(primary_record(100, ptr0))
    got = bt.run()
    n_ok = min(links, ao.MAX_DEPTH + 1)
    assert len(got) == n_ok + (1 if links > ao.MAX_DEPTH + 1 else 0)
    for d in range(n_ok):
        r = got[d]
        assert r["depth"] == d and r["parent"] == (0 if d == 0 else d - 1)
        check_decoded(r, chans[d], pdus[d])
        assert abs(int(r["sample_index"]) - starts[d]) == 0
    if links > ao.MAX_DEPTH + 1:
        assert got[-1]["status"] == ao.DEPTH_LIMIT and got[-1]["depth"] == ao.MAX_DEPTH + 1


def test_chain_pointing_back_at_itself_ends():
    rng = np.random.default_rng(5)
    bt = Batch(20000, seed=5)
    starts, pdus, ptr0 = _chain(bt, rng, 100, [4, 9], [0, 1], loop_last=True)
    bt.frames.append(primary_record(100, ptr0))
    got = bt.run()
    assert len(got) == 3
    check_decoded(got[2], 9, pdus[1])
    assert got[2]["sample_index"] == got[1]["sample_index"] and got[2]["first"] == 1 and got[2]["parent"] == 1


def test_three_primaries_one_packet():
    """37 / 38 / 39 point at one AUX_ADV_IND: every pointer finds it, `first` names the earliest, the chain is followed once."""
    rng = np.random.default_rng(9)
    bt = Batch(40000, seed=9)
    starts, pdus, _ = _chain(bt, rng, 9000, [17, 2], [1, 0])
    for j, s in enumerate((1000, 4000, 7000)):
        off = (starts[0] - s) // 4 // 30
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(17, 0, 30, off, 1), channel=37 + j))
    got = bt.run()
    assert len(got) == 4
    assert list(got["depth"]) == [0, 0, 0, 1] and list(got["parent"]) == [0, 1, 2, 0]
    assert list(got["first"]) == [0, 0, 0, 3]
    for r in got[:3]:
        check_decoded(r, 17, pdus[0])
    check_decoded(got[3], 2, pdus[1])


def test_shard_coordinates():
    """A shard reports whole-capture indices; windows that leave its buffer are OUTSIDE there."""
    rng = np.random.default_rng(11)
    whole = Batch(60000, seed=11)
    pdu = aux_pdu(rng, 60)
    s = 20000
    at = s + ao.window(30, 30, 1)[0] + 20
    plant_stride(whole.b[6], at, aux_symbols(6, pdu), 4)
    whole.frames.append(primary_record(s, synth.aux_ptr_bytes(6, 1, 30, 30, 0)))
    want = whole.run()
    check_decoded(want[0], 6, pdu)
    pre, w0 = 128, 2                                              # buffer = capture samples [8192 * 2 - 128, ...)
    hi = s + ao.window(30, 30, 1)[1]
    for end, status in ((60000, None), (at + 900, ao.TRUNCATED), (hi + 100, ao.OUTSIDE)):
        sh = Batch(end - (8192 * w0 - pre))
        for c in list(whole.b):
            sh.b[c] = whole.b[c][8192 * w0 - pre:end]
        sh.frames = whole.frames
        got = sh.run(first_window=w0, pre_out=pre)
        if status is None:
            assert got.tobytes() == want.tobytes()
        else:
            assert got[0]["status"] == status


# ------------------------------------------------------------------------------------------------ end to end (CPU)
def _taps(name):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from gen_tables import PFB_DESIGNS, kaiser_lowpass
    return kaiser_lowpass(*PFB_DESIGNS[name])


def end_to_end(oracle_mod, cap, taps_name: str):
    """numpy capture -> the channelizer's definition (pfb_oracle) -> quantiser and slicer -> the BLE oracle on 37..39 ->
    aux_oracle.  Returns (aux list, recovered fraction of the injected aux packets)."""
    bins = [chanplan.ble_channel_bin(c) for c in range(40)]
    y = oracle_mod.pfb(cap.iq, _taps(taps_name), bins, fast=True)
    n = y.shape[1]
    b = np.zeros((40, n), np.uint8)
    frames = []
    for c in range(40):
        q = oracle_mod.ble_quantize(y[c], 100.0).astype(np.int64).reshape(-1, 2)
        nxt = np.vstack([q[1:], np.zeros((1, 2), np.int64)])
        b[c] = (q[:, 0] * nxt[:, 1] - nxt[:, 0] * q[:, 1] > 0)
        if c >= 37:
            fr = oracle_mod.ble_decode(q.astype(np.int8), c)
            fr["channel"] = c
            frames.append(fr)
    fr = np.concatenate(frames)
    words = np.stack([pack_words(b[c], n_words=4 + (n + 31) // 32 + 64) for c in range(40)])[None]
    aux = ao.aux_list(words, fr, n)
    return aux, recall(aux, cap.meta["aux"])


def recall(aux, truth) -> float:
    """Fraction of the injected packets decoded with a good CRC.  Where a packet is found, every pointer to it found it, at its
    place: the offsets from the nominal AA bit 0 are the filters' delay (the same for every packet of a PHY) within a sample."""
    got = {(int(r["channel"]), bytes(r["bytes"][: int(r["len"])])) for r in aux if r["status"] == ao.OK and r["crc_ok"]}
    found = sum((t.channel, t.data) in got for t in truth)
    for phy in (0, 1):
        d = [int(r["sample_index"]) - t.anchor for t in truth if t.phy == phy for r in aux
             if r["status"] == ao.OK and bytes(r["bytes"][: int(r["len"])]) == t.data]
        assert not d or max(d) - min(d) <= 2, d
    return found / len(truth)


@pytest.mark.parametrize("taps", ["BLE_384", "BLE_768"])
@pytest.mark.parametrize("esn0", [None, 25.0])
def test_end_to_end_recall(oracle_mod, taps, esn0):
    cap = synth.ext_adv_capture(seconds=0.09, seed=9100, esn0_db=esn0, n_events=4, max_chain=2, data_len=(0, 200))
    truth = cap.meta["aux"]
    assert {t.phy for t in truth} == {0, 1} and max(t.depth for t in truth) >= 1
    aux, rec = end_to_end(oracle_mod, cap, taps)
    assert rec == 1.0, (taps, esn0, rec)


# ------------------------------------------------------------------------------------------------ host side
def _aux_of_chain():
    rng = np.random.default_rng(21)
    bt = Batch(40000, seed=21)
    starts, pdus, _ = _chain(bt, rng, 9000, [17, 2, 30], [1, 0, 1])
    for j, s in enumerate((1000, 4000)):
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(17, 0, 30, (starts[0] - s) // 4 // 30, 1), channel=37 + j))
    return bt.run().astype(_abi.AUX_DTYPE), pdus


def test_ext_adv_parsing_and_chain_reassembly():
    aux, pdus = _aux_of_chain()
    msgs = messages.ble_ext_adv(aux)
    assert [m["index"] for m in msgs] == [0, 2, 3]                 # entry 1 found the same packet as entry 0
    root = msgs[0]
    f = messages._ext_fields(pdus[0] + synth.ble_crc24(pdus[0]))
    hl = pdus[0][2] & 0x3F
    assert root["adv_a"] == bytes(pdus[0][4:10])[::-1].hex() and root["tx_power"] == -7 and root["phy"] == "2M"
    assert root["did"] == int.from_bytes(pdus[0][10:12], "little") & 0xFFF and root["adv_data"] == pdus[0][3 + hl:]
    assert f["adv_data"] == root["adv_data"]
    assert root["chain"] == [0, 2, 3] and root["complete"]
    assert root["chain_data"] == b"".join(p[3 + (p[2] & 0x3F):] for p in pdus)
    broken = aux.copy()
    broken[3]["crc_ok"] = 0
    assert messages.ble_ext_adv(broken)[0]["complete"] is False


def test_pcap_aux_block_bytes():
    aux, pdus = _aux_of_chain()
    blob = formats.ble_pcap_aux_block(aux)
    at, recs = 0, []
    while at < len(blob):
        n = struct.unpack(">i", blob[at + 8:at + 12])[0]
        recs.append(blob[at + 16:at + 16 + n])
        at += 16 + n
    assert len(recs) == 3
    for k, rec in zip((0, 2, 3), recs):
        r = aux[k]
        flags = struct.unpack("<H", rec[8:10])[0]
        assert rec[0] == r["channel"] and rec[1:8] == b"\0" * 7
        assert flags == 0x0001 | (1 << 7) | (int(r["phy"]) << 14)
        assert struct.unpack("<I", rec[10:14])[0] == ADV_AA and rec[14:] == bytes(r["bytes"][: int(r["len"]) - 3])


class AuxEngine(RecordingEngine):
    aux = None

    def ble_aux(self):
        return self.aux


def test_cli_aux(tmp_path):
    aux, _ = _aux_of_chain()
    out = io.StringIO()
    assert btle_cli.run(btle_cli.parse_commandline(["--aux", "--iq", "-"], out=out), out=out) == 1
    assert "--aux needs --wideband" in out.getvalue()
    pcap = tmp_path / "x.pcap"
    AuxEngine.aux = aux
    out = io.StringIO()
    o = btle_cli.parse_commandline(["--wideband", "--aux", "-s", str(pcap)], out=out)
    blk = np.zeros(24 * 8192, np.complex64)
    rc = btle_cli.run(o, out=out, engine_factory=lambda mode, **kw: AuxEngine(mode, **{k: v for k, v in kw.items() if k == "max_samples"}),
                      blocks=[blk])
    assert rc == 0
    lines = [ln for ln in out.getvalue().splitlines() if ln.startswith("AUX ")]
    assert len(lines) == 3 and all(len(ln.split()) == 8 for ln in lines)
    m = messages.ble_ext_adv(aux)[0]
    assert lines[0] == f"AUX Ch17 PHY2M AdvA:{m['adv_a']} ADI:{m['did']:03x}/{m['sid']:x} Depth0 PloadL{m['pload_len']} CRC0"
    data = pcap.read_bytes()
    assert data.startswith(formats.PCAP_HDR_BLE) and data.endswith(formats.ble_pcap_aux_block(aux))
