"""BLE periodic advertising (snrx_ble_periodic): CSA#2 against the Core specification's sample data, the contract's
restatement (oracle/periodic_oracle.py) against the kernels' host-side cores (tests/emu/emu_sync.cu), constructed bit
streams that put each edge of the contract on the oracle, end to end through the channelizer's CPU statement, and the host
side (messages, lines, pcap, CLI).  No GPU."""
from __future__ import annotations

import ctypes
import functools
import io
import os
import shutil
import struct
import subprocess
from typing import Callable, NamedTuple

import numpy as np
import pytest

import ble_bits as bb
from fake_engine import RecordingEngine
from oracle import aux_oracle as ao
from oracle import periodic_oracle as po
from snout_b200 import _abi, btle_cli, formats, messages, synth
from test_ble_aux import Batch, aux_symbols, plant_stride, primary_record

N_CH = 40
KAT_AA = 0x8E89BED6                                   # Core Vol 6 Part C 3 (CSA#2 sample data)
KAT_NINE = [9, 10, 21, 22, 23, 33, 34, 35, 36]


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sync_emu(tmp_path_factory):
    """tests/emu/emu_sync.cu (the cores of snout_b200/csrc/ble_sync.cuh) built with the flags of tests/emu/Makefile into a
    temporary directory."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = str(tmp_path_factory.mktemp("emu_sync") / "libemu_sync.so")
    r = subprocess.run([nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr",
                        "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-o", out,
                        os.path.join(ROOT, "tests", "emu", "emu_sync.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = ctypes.CDLL(out)
    lib.emu_csa2_channel.restype = ctypes.c_int
    lib.emu_crc_seed_of.restype = ctypes.c_uint32
    return lib


# ------------------------------------------------------------------------------------------------ CSA#2
def _chm(used) -> int:
    return sum(1 << c for c in used)


def test_csa2_known_answers(sync_emu):
    assert ((KAT_AA >> 16) ^ KAT_AA) & 0xFFFF == 0x305F
    for used, pairs in ((list(range(37)), [(0, 25), (1, 20), (2, 6), (3, 21)]), (KAT_NINE, [(6, 23), (7, 9), (8, 34)])):
        for counter, ch in pairs:
            assert po.csa2(counter, KAT_AA, used) == ch
            assert synth.csa2_channel(counter, KAT_AA, used) == ch
            assert sync_emu.emu_csa2_channel(ctypes.c_uint32(counter), ctypes.c_uint32(KAT_AA), ctypes.c_uint64(_chm(used))) == ch


@pytest.mark.parametrize("aa,used", [(0x8E89BED6, KAT_NINE), (0x5A3C9E71, [0, 36]), (0x12345678, list(range(0, 37, 3))),
                                     (0xFFFF0000, list(range(37))), (0x0000FFFF, [5, 17, 18, 30])])
def test_csa2_kernel_equals_oracle_on_every_counter(sync_emu, aa, used):
    chm = ctypes.c_uint64(_chm(used))
    got = [sync_emu.emu_csa2_channel(ctypes.c_uint32(c), ctypes.c_uint32(aa), chm) for c in range(65536)]
    want = [po.csa2(c, aa, used) for c in range(65536)]
    assert got == want
    assert [synth.csa2_channel(c, aa, used) for c in range(0, 65536, 97)] == want[::97]
    assert set(got) <= set(used)


# ------------------------------------------------------------------------------------------------ windows and listed events
def _si(offset=517, units=30, adjust=0, interval=6, sca=0, used=range(37), aa=0x5A3C9E71, crc_init=0x123456, pa=100):
    return po.SyncInfo(synth.sync_info_bytes(offset, units, interval, _chm(used), sca, aa, crc_init, pa, adjust))


def _emu_window(sync_emu, si, k):
    lo, hi = ctypes.c_int64(), ctypes.c_int64()
    sync_emu.emu_sync_window(si.offset, si.units_us, si.adjust, si.interval, si.sca, ctypes.c_int64(k), ctypes.byref(lo), ctypes.byref(hi))
    return lo.value, hi.value


def _emu_range(sync_emu, si, s, sps, base, n_out):
    a, b = ctypes.c_int64(), ctypes.c_int64()
    sync_emu.emu_sync_k_range(si.offset, si.units_us, si.adjust, si.interval, si.sca, ctypes.c_int64(s), sps, ctypes.c_int64(base),
                         ctypes.c_int64(n_out), ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def test_window_floor_and_ceiling_at_negative_d(sync_emu):
    si = _si(offset=517, sca=0)                       # O = 15 510 us, I' = 7500 us, p = 500
    d_lo, d_hi = 15510 - 3 * 7500, 15510 + 30 - 3 * 7500
    assert d_lo == -6990 and d_hi == -6960
    lo, hi = po.window(si, -3)
    assert lo == -27974 - 8 and hi == -27826 + 8       # floor(-27 973.98), ceil(-27 826.08): not C's truncation
    # C's truncating division: one sample later at the low end, and aux_window's (a + 999999) / 10^6 one sample early at the
    # high end
    assert int(4 * d_lo * 1000500 / 10**6) - 8 == lo + 1 and int((4 * d_hi * 999500 + 999999) / 10**6) + 8 == hi + 1
    assert _emu_window(sync_emu, si, -3) == (lo, hi)
    # k = 0 is aux_window with ppm from the SCA
    for sca, ca in ((0, 0), (5, 1)):
        s2 = _si(offset=517, sca=sca)
        assert po.window(s2, 0) == ao.window(30, 517, ca)


def test_kernel_window_and_range_equal_the_oracle(sync_emu):
    rng = np.random.default_rng(5)
    for _ in range(300):
        si = _si(offset=int(rng.integers(1, 8192)), units=int(rng.choice([30, 300])), adjust=int(rng.integers(0, 2)),
                 interval=int(rng.integers(6, 400)), sca=int(rng.integers(0, 8)))
        for k in rng.integers(-3000, 3000, 5):
            assert _emu_window(sync_emu, si, int(k)) == po.window(si, int(k))
        sps = int(rng.choice([2, 4]))
        s = int(rng.integers(0, 4_000_000))
        base = int(rng.integers(-2_000_000, s + 1))
        n_out = int(rng.integers(2, 6_000_000))
        r = po.listed_range(si, s, sps, base, n_out)
        got = _emu_range(sync_emu, si, s, sps, base, n_out)
        assert (got[0], got[1] + 1) == ((r.start, r.stop) if len(r) else (got[0], got[0])), (got, r)
        if not len(r):
            assert got[1] < got[0]


def test_rule_a_last_listed_and_first_unlisted(sync_emu):
    """A buffer long enough to reach rule (a)'s edge on both sides: the last listed k has a window of at most half the
    interval, the next one does not."""
    for sca, interval, units in ((0, 6, 30), (0, 9, 300), (7, 6, 30)):
        si = _si(offset=4000, units=units, interval=interval, sca=sca)
        r = po.listed_range(si, 10**12, 4, 0, 2 * 10**12)
        for k, inside in ((r.start, True), (r.start - 1, False), (r.stop - 1, True), (r.stop, False)):
            lo, hi = po.window(si, k)
            assert (hi - lo + 1 <= 2500 * interval) == inside
        assert _emu_range(sync_emu, si, 10**12, 4, 0, 2 * 10**12) == (r.start, r.stop - 1)


def test_listed_events_are_contiguous_and_disjoint():
    """The contract's bound, swept: for any SyncInfo, the window width grows by at least 8 I' p / 10^6 >= 1.2 samples per
    event away from D = 0, more than the two roundings (less than 2 samples together) can take back, so rule (a) holds on one
    contiguous range of k; and a window of at most 2500 Interval samples plus the 31 sps access-address span ends before
    the next event's window starts (the windows' centres are 5000 Interval (1 -+ p) samples apart)."""
    rng = np.random.default_rng(2024)
    for _ in range(20000):
        si = _si(offset=int(rng.integers(1, 8192)), units=int(rng.choice([30, 300])), adjust=int(rng.integers(0, 2)),
                 interval=int(rng.integers(6, 201)), sca=int(rng.integers(0, 8)))
        kc = -(si.o_us // (1250 * si.interval))
        ks = [k for k in range(kc - 12, kc + 13) if po.rule_a(si, k)]
        assert ks == list(range(ks[0], ks[-1] + 1))
        for k in ks[:-1]:
            assert po.window(si, k)[1] + 31 * 4 < po.window(si, k + 1)[0]
    # at the far edges too
    for sca in range(8):
        si = _si(interval=6, sca=sca, units=300)
        r = po.listed_range(si, 10**13, 4, 0, 2 * 10**13)
        for k in (r.start, r.stop - 2):
            assert po.window(si, k)[1] + 31 * 4 < po.window(si, k + 1)[0]


# ------------------------------------------------------------------------------------------------ SyncInfo parsing
def test_sync_info_parsing(sync_emu):
    si_b = synth.sync_info_bytes(8191, 300, 65535, _chm(KAT_NINE), 7, 0xA1B2C3D4, 0xABCDEF, 0xFFFE, adjust=1)
    assert si_b[13:16] == bytes([0xAB, 0xCD, 0xEF])            # c0 sent first
    for fields in ((b"\1" * 6, None, None), (b"\1" * 6, 0x1234, synth.aux_ptr_bytes(3, 1, 30, 9, 0)), (None, None, None)):
        adv_a, adi, ptr = fields
        pdu = synth.ext_pdu(synth.ext_header(0, adv_a, 0, adi, ptr, -3, sync_info=si_b, acad=b"\2\x2c\0"), b"data")
        si = po.parse_sync_info(pdu, pdu[1])
        assert (si.offset, si.units_us, si.adjust, si.interval, si.sca, si.aa, si.crc_init, si.pa_counter) == \
            (8191, 300, 1, 65535, 7, 0xA1B2C3D4, 0xABCDEF, 0xFFFE)
        assert si.used == KAT_NINE and si.o_us == 8191 * 300 + 2_457_600 and si.valid()
        f = (ctypes.c_int32 * 9)()
        chm = ctypes.c_uint64()
        buf = np.frombuffer(pdu, np.uint8).copy()
        assert sync_emu.emu_sync_info_parse(buf.ctypes.data_as(ctypes.c_void_p), pdu[1], f, ctypes.byref(chm)) == 0
        assert list(f) == [8191, 300, 1, 65535, 7, ctypes.c_int32(0xA1B2C3D4).value, 0xABCDEF, 0xFFFE, 1] and chm.value == _chm(KAT_NINE)
        d = messages.sync_info_fields(si_b)
        assert d["channels"] == KAT_NINE and d["crc_init"] == 0xABCDEF and d["ppm"] == 20 and d["offset_us"] == si.o_us
    # one byte short of the SyncInfo, no flag, and the SyncInfo values that describe no train
    pdu = synth.ext_pdu(synth.ext_header(0, b"\1" * 6, 0, None, None, None, sync_info=si_b))
    short = bytes([pdu[0], pdu[1] - 1, pdu[2] - 1]) + pdu[3:-1]
    assert po.parse_sync_info(short, short[1]) is None
    assert po.parse_sync_info(synth.ext_pdu(synth.ext_header(0, b"\1" * 6)), 8) is None
    for kw in (dict(offset=0), dict(interval=5), dict(used=[4])):
        assert not _si(**kw).valid()
    assert _si(interval=6, used=[4, 5]).valid()
    assert sync_emu.emu_crc_seed_of(ctypes.c_uint32(0xABCDEF)) == bb.crc_internal(synth.sync_crc_seed(0xABCDEF)) == bb.crc_internal(0xEFCDAB)


def ext_header_sweep(seed):
    """(buffer, n_payload, flags, hlen) for every flags byte, every extended header length 0..63 and payloads of hlen,
    hlen + 1 and hlen + 2 bytes: a PDU of type 7 with seeded random bytes everywhere else.  The buffer always holds the
    header length and flags bytes, whatever n_payload says."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, (256, 64, 3, 2 + 65), dtype=np.uint8)
    for flags in range(256):
        for hlen in range(64):
            for j, n_payload in enumerate((hlen, hlen + 1, hlen + 2)):
                buf = noise[flags, hlen, j, : 2 + max(n_payload, 2)].copy()
                buf[0] = (buf[0] & 0xF0) | 7
                buf[1] = n_payload
                buf[2] = (buf[2] & 0xC0) | hlen
                buf[3] = flags
                yield buf, n_payload, flags, hlen


def test_aux_ptr_and_sync_info_parse_on_every_header(sync_emu):
    """The kernels' AuxPtr and SyncInfo parsers equal the oracles' on every flags byte and header length, including the
    headers too short for the field and the payloads too short for the header."""
    fa, fs, chm = (ctypes.c_int32 * 5)(), (ctypes.c_int32 * 9)(), ctypes.c_uint64()
    n_aux = n_sync = 0
    for buf, n_payload, flags, hlen in ext_header_sweep(20261):
        ptr, pdu = buf.ctypes.data_as(ctypes.c_void_p), buf.tobytes()
        want = ao.parse_aux_ptr(pdu, n_payload)
        rc = sync_emu.emu_aux_ptr_parse(ptr, n_payload, fa)
        assert (rc == 0) == (want is not None), (flags, hlen, n_payload)
        if want is not None:
            assert tuple(fa) == want, (flags, hlen, n_payload)
            n_aux += 1
        si = po.parse_sync_info(pdu, n_payload)
        rc = sync_emu.emu_sync_info_parse(ptr, n_payload, fs, ctypes.byref(chm))
        assert (rc == 0) == (si is not None), (flags, hlen, n_payload)
        if si is not None:
            assert list(fs) == [si.offset, si.units_us, si.adjust, si.interval, si.sca, ctypes.c_int32(si.aa).value, si.crc_init,
                                si.pa_counter, int(si.valid())] and chm.value == si.chm, (flags, hlen, n_payload)
            n_sync += 1
    assert n_aux > 10000 and n_sync > 1000                      # both parsers find their field on a good share of the sweep


# ------------------------------------------------------------------------------------------------ constructed streams
class Train:
    """A periodic-advertising train's SyncInfo and the symbols of its packets."""

    def __init__(self, aa=0x5A3C9E71, crc_init=0x3C2B1A, interval=6, used=range(37), sca=0, pa=100, offset=517, units=30,
                 adjust=0, phy=0):
        self.aa, self.crc_init, self.phy, self.pa = aa, crc_init, phy, pa
        self.used = list(used)
        self.sps = 2 if phy else 4
        self.bytes = synth.sync_info_bytes(offset, units, interval, _chm(self.used), sca, aa, crc_init, pa, adjust)
        self.si = po.SyncInfo(self.bytes)

    def window(self, k):
        return po.window(self.si, k)

    def channel(self, k):
        return po.csa2((self.pa + k) % 65536, self.aa, self.used)

    def symbols(self, k, pdu, crc_ok=True):
        return bb.frame_symbols(self.channel(k), pdu[:2], pdu[2:], crc_ok, aa=self.aa, crc_init=synth.sync_crc_seed(self.crc_init))


def sync_pdu(rng, n=20, acad=b"", chained=False) -> bytes:
    ptr = synth.aux_ptr_bytes(7, 1, 30, 40, 0) if chained else None
    return synth.ext_pdu(synth.ext_header(0, None, 0, None, ptr, None, acad=acad), bytes(rng.integers(0, 256, n, dtype=np.uint8)))


class Scene:
    """One capture's bit streams: AUX_ADV_INDs with a SyncInfo, the ADV_EXT_IND records pointing at them, and the events."""

    def __init__(self, n, seed=0):
        self.bt = Batch(n, seed=seed)
        for c in (37, 38, 39):
            self.bt.b[c] &= 0
        self.rng = np.random.default_rng(seed + 1)

    def source(self, tr: Train, s: int, ch: int = 20, prim_channel: int = 37, gap: int = 2400, adv_a=b"\1\2\3\4\5\6"):
        pdu = synth.ext_pdu(synth.ext_header(0, adv_a, 0, 0x1234, None, None, sync_info=tr.bytes))
        plant_stride(self.bt.b[ch], s, aux_symbols(ch, pdu), tr.sps)
        ps = s - gap
        self.bt.frames.append(primary_record(ps, synth.aux_ptr_bytes(ch, 1, 30, gap // 4 // 30, tr.phy), channel=prim_channel))
        return pdu

    def event(self, tr: Train, s: int, k: int, at: int, n: int = 20, crc_ok=True, **kw) -> bytes:
        """The event-k packet of a train whose source is at s, AA bit 0 at s + at."""
        pdu = sync_pdu(self.rng, n, **kw)
        plant_stride(self.bt.b[tr.channel(k)], s + at, tr.symbols(k, pdu, crc_ok), tr.sps)
        return pdu


class SCase(NamedTuple):
    name: str
    words: np.ndarray                     # uint32 [captures, 40, words]
    n_out: int
    frames: np.ndarray                    # the ADV_EXT_IND records the construction means
    spots: tuple                          # (capture, channel, s) of the planted ADV_EXT_INDs
    check: Callable                       # the expectation on the oracle's list
    shard: tuple | None = None            # (pre_out, first_window, n_windows)
    first_capture: int = 0

    def geo(self) -> dict:
        pre, w0, _ = self.shard or (0, 0, 0)
        return dict(first_window=w0, pre_out=pre, first_capture=self.first_capture)

    def shard_arg(self) -> dict:
        pre, w0, nw = self.shard or (0, 0, 0)
        return dict(pre_samples=24 * pre, body_samples=24 * 8192 * nw, first_window=w0, first_capture_id=self.first_capture)

    def lists(self, frames=None):
        aux = ao.aux_list(self.words, self.frames if frames is None else frames, self.n_out, **self.geo())
        return aux, po.sync_list(self.words, aux, self.n_out, **self.geo())


def case(name, scenes, check, shard=None, first_capture=0) -> SCase:
    """Every ADV_EXT_IND record is planted as a real frame at its sample_index, so that the engine's own poll provides it; the
    last decision of every stream is 0, as the front end leaves it."""
    scenes = scenes if isinstance(scenes, list) else [scenes]
    base = 8192 * shard[1] - shard[0] if shard else 0
    spots, frames = [], []
    for cap, sc in enumerate(scenes):
        for f in sc.bt.frames:
            s, ch = int(f["sample_index"]), int(f["channel"])
            pdu = bytes(f["bytes"][: int(f["len"]) - 3])
            plant_stride(sc.bt.b[ch], s - base, bb.frame_symbols(ch, pdu[:2], pdu[2:]), 4)
            spots.append((cap, ch, s))
            g = f.copy()
            g["capture_id"] = first_capture + cap
            frames.append(g)
    w = np.concatenate([sc.bt.words() for sc in scenes])
    n = scenes[0].bt.n
    w[:, :, 4 + (n - 1) // 32] &= ~np.uint32(1 << ((n - 1) % 32))
    fr = np.array(frames, dtype=_abi.FRAME_DTYPE)
    fr = fr[np.lexsort((fr["sample_index"], fr["channel"], fr["capture_id"]))]
    return SCase(name, w, n, fr, tuple(spots), check, shard, first_capture)


def ev(got, k, source=None):
    sel = got["event"] == k
    if source is not None:
        sel &= got["source"] == source
    (r,) = got[sel]
    return r


def found(r, tr: Train, at: int, pdu: bytes, k: int, crc_ok=True):
    want = pdu + synth.ble_crc24(pdu, synth.sync_crc_seed(tr.crc_init))
    assert r["status"] == po.OK and int(r["sample_index"]) == at and r["channel"] == tr.channel(k)
    assert r["len"] == len(want) and bool(r["crc_ok"]) == crc_ok and (not crc_ok or bytes(r["bytes"][: len(want)]) == want)
    assert r["access_addr"] == tr.aa and r["crc_init"] == tr.crc_init and r["event_counter"] == (tr.pa + k) % 65536


def _window_edges():
    out = []
    tr = Train(offset=517, sca=0)
    s = 60_000
    for k in (-3, 2):
        lo, hi = tr.window(k)
        for name, at, hit in (("lo-1", lo - 1, False), ("lo", lo, True), ("hi", hi, True), ("hi+1", hi + 1, False)):
            sc = Scene(s + 4 * (15510 + 3 * 7500) + 6000, seed=abs(k) * 10 + len(name))
            sc.source(tr, s)
            pdu = sc.event(tr, s, k, at)

            def check(got, k=k, at=at, hit=hit, pdu=pdu):
                r = ev(got, k)
                assert (int(r["win_lo"]), int(r["win_hi"])) == (s + tr.window(k)[0], s + tr.window(k)[1])
                if hit:
                    found(r, tr, s + at, pdu, k)
                else:
                    assert r["status"] == po.NOT_FOUND and r["sample_index"] == -1
            out.append(case(f"edge_k{k}_{name}", sc, check))
    return out


def _buffer_ends():
    """OUTSIDE at both ends, the first and last listed events, and TRUNCATED / OK at the end."""
    out = []
    for sps, phy in ((4, 0), (2, 1)):
        tr = Train(offset=517, sca=0, phy=phy)
        lo3, hi3 = tr.window(-3)
        for d, want in ((0, "searched"), (-1, "outside")):
            s = -lo3 + d                                # win_lo(-3) = d
            sc = Scene(s + 40_000, seed=d + sps)
            sc.source(tr, s)

            def check(got, tr=tr, d=d, want=want, s=s):
                r = ev(got, -3)
                assert int(r["win_lo"]) == d
                assert (r["status"] == po.OUTSIDE) == (want == "outside")
                assert got["event"].min() == -3                      # win_hi(-4) + 31 sps < 0: not listed
                assert s + tr.window(-4)[1] + 31 * sps < 0
            out.append(case(f"start_{sps}_{want}", sc, check))
        s = 40_000
        lo1, hi1 = tr.window(1)
        for n, want in ((s + hi1 + 31 * sps + 2, "searched"), (s + hi1 + 31 * sps + 1, "outside"), (s + lo1 + 2, "lo_last"),
                        (s + lo1 + 1, "unlisted")):
            sc = Scene(n, seed=n)
            sc.source(tr, s)

            def check(got, tr=tr, want=want, n=n):
                if want == "unlisted":
                    assert got["event"].max() == 0
                    return
                r = ev(got, 1)
                assert (r["status"] == po.OUTSIDE) == (want in ("outside", "lo_last"))
                if want == "lo_last":
                    assert int(r["win_lo"]) == n - 2
            out.append(case(f"end_{sps}_{want}", sc, check))
        pdu_len = 40
        at = hi1 - 4
        nbits = 32 + 8 * (2 + pdu_len + 3)
        end = s + at + (nbits - 1) * sps
        for n, status in ((end + 2, po.OK), (end + 1, po.TRUNCATED), (s + at + 47 * sps + 1, po.TRUNCATED)):
            if s + hi1 + 31 * sps > n - 2:
                continue
            sc = Scene(n, seed=n)
            sc.source(tr, s)
            sc.event(tr, s, 1, at, n=pdu_len - 2)

            def check(got, tr=tr, status=status):
                r = ev(got, 1)
                assert r["status"] == status and int(r["sample_index"]) == s + at
            out.append(case(f"trunc_{sps}_{n - end}", sc, check))
    return out


def _phases_wrap_remap():
    out = []
    for phase in (0, 1):
        tr = Train(offset=300, sca=3, phy=1, interval=7)
        s = 30_001
        sc = Scene(s + 4 * (9000 + 3 * 8750) + 4000, seed=phase)
        sc.source(tr, s)
        pdus = {k: (tr.window(k)[0] + 11 + phase - (s % 2), sc.event(tr, s, k, tr.window(k)[0] + 11 + phase - (s % 2), n=30))
                for k in (-1, 0, 2)}

        def check(got, tr=tr, pdus=pdus, s=s):
            for k, (at, pdu) in pdus.items():
                r = ev(got, k)
                found(r, tr, s + at, pdu, k)
                assert r["phase"] == (s + at) % 2 and r["phy"] == ao.PHY_2M
        out.append(case(f"2m_phase{phase}", sc, check))
    for pa, ks in ((65535, (0, 1, 2)), (0, (-2, -1, 0))):
        tr = Train(pa=pa, used=KAT_NINE, aa=0x8E89BED7, interval=6)
        s = 70_000
        sc = Scene(s + 4 * (15510 + 3 * 7500) + 4000, seed=pa % 7)
        sc.source(tr, s)
        pdus = {k: sc.event(tr, s, k, tr.window(k)[0] + 9) for k in ks}

        def check(got, tr=tr, pdus=pdus, s=s):
            for k, pdu in pdus.items():
                found(ev(got, k), tr, s + tr.window(k)[0] + 9, pdu, k)
            counters = {int(ev(got, k)["event_counter"]) for k in pdus}
            assert {0, 65535} <= counters
        out.append(case(f"wrap_{pa}", sc, check))
    # remapped channels: events whose unmapped channel is not used
    tr = Train(used=[2, 11, 29], aa=0x71764129, pa=4000)
    s = 60_000
    sc = Scene(s + 4 * (15510 + 4 * 7500) + 4000, seed=9)
    sc.source(tr, s)
    pdus = {k: sc.event(tr, s, k, tr.window(k)[1] - 3) for k in (-1, 0, 1, 2, 3)}

    def check_remap(got, tr=tr, s=s):
        cid = ((tr.aa >> 16) ^ tr.aa) & 0xFFFF
        for k, pdu in pdus.items():
            found(ev(got, k), tr, s + tr.window(k)[1] - 3, pdu, k)
        assert sum(tr.channel(k) != _unmapped(tr.pa + k, cid) for k in pdus) >= 3
    out.append(case("remap", sc, check_remap))
    return out


def _unmapped(counter, cid):
    u = (counter % 65536) ^ cid
    for _ in range(3):
        u = int(f"{u & 0xFF:08b}"[::-1], 2) | (int(f"{u >> 8:08b}"[::-1], 2) << 8)
        u = (17 * u + cid) & 0xFFFF
    return (u ^ cid) % 37


def _sources_and_warps():
    out = []
    # two AUX_ADV_INDs of one AA at the same sample on different channels (the lower list index is the source), and a
    # third AA-sharing one later; a second train whose events sit next to the first's in the list (one warp each)
    a = Train(offset=600, pa=10)
    a_late = Train(offset=500, pa=10)
    b = Train(aa=0x3F1E2D4C, crc_init=0xA5A5A5, offset=900, pa=500, units=300, sca=2, used=range(0, 37, 2))
    s = 40_000
    sc = Scene(s + 12_000 + 4 * (900 * 300 + 2 * 7500) + 4000, seed=3)
    sc.source(a, s, ch=5, prim_channel=37)
    sc.source(a_late, s, ch=6, prim_channel=38)
    sc.source(a_late, s + 5000, ch=8, prim_channel=39)
    sc.source(b, s + 12_000, ch=30, prim_channel=39, gap=6000)
    pa = {k: sc.event(a, s, k, a.window(k)[0] + 12) for k in (0, 1)}
    lo, hi = b.window(0)
    assert hi - lo > 1024 + 64                             # the window spans two 32-word passes; the packet is in the second
    pb = {k: sc.event(b, s + 12_000, k, b.window(k)[1] - 2) for k in (0, 1)}

    def check(got):
        srcs = sorted(set(got["source"].tolist()))
        assert len(srcs) == 2
        ga = got[got["source"] == srcs[0]]
        gb = got[got["source"] == srcs[1]]
        assert (ga["access_addr"] == a.aa).all() and (gb["access_addr"] == b.aa).all()
        for k, pdu in pa.items():
            found(ev(ga, k), a, s + a.window(k)[0] + 12, pdu, k)     # predicted from the first source, not a_late's
        for k, pdu in pb.items():
            found(ev(gb, k), b, s + 12_000 + b.window(k)[1] - 2, pdu, k)
    out.append(case("equal_sources_two_trains", sc, check))
    return out


def _captures_and_shards():
    out = []
    tr = Train(offset=517, pa=7)
    s = 50_000
    n = s + 4 * (15510 + 2 * 7500) + 4000
    scenes, pdus = [], []
    for cap in range(3):
        sc = Scene(n, seed=40 + cap)
        if cap != 1:
            sc.source(tr, s + 100 * cap)
            pdus.append(sc.event(tr, s + 100 * cap, 1, tr.window(1)[0] + 20 + cap))
        scenes.append(sc)

    def check(got, s=s):
        assert sorted(set(got["capture_id"].tolist())) == [5, 7]
        for cap, pdu in zip((0, 2), pdus):
            g = got[got["capture_id"] == 5 + cap]
            found(ev(g, 1), tr, s + 100 * cap + tr.window(1)[0] + 20 + cap, pdu, 1)
    out.append(case("three_captures", scenes, check, first_capture=5))
    # a shard: buffer = capture samples [8192 w0 - pre, ...); whole-capture indices
    w0, pre = 3, 128
    base = 8192 * w0 - pre
    s = base + 40_000
    sc_whole = Scene(s + 4 * (15510 + 2 * 7500) + 4000, seed=77)
    sc_whole.source(tr, s)
    p = {k: sc_whole.event(tr, s, k, tr.window(k)[0] + 30) for k in (-1, 0, 1)}
    sh = Scene(sc_whole.bt.n - base, seed=78)
    for c in list(sc_whole.bt.b):
        sh.bt.b[c] = sc_whole.bt.b[c][base:].copy()
    sh.bt.frames = [f.copy() for f in sc_whole.bt.frames]

    def check_shard(got):
        for k, pdu in p.items():
            found(ev(got, k), tr, s + tr.window(k)[0] + 30, pdu, k)
        assert (got["win_hi"] + 31 * 4 >= base).all() and (got["win_lo"] <= base + sh.bt.n - 2).all()
    out.append(case("shard", sh, check_shard, shard=(pre, w0, (sh.bt.n - pre) // 8192)))
    return out


def all_cases() -> list[SCase]:
    cases = []
    for f in (_window_edges, _buffer_ends, _phases_wrap_remap, _sources_and_warps, _captures_and_shards):
        cases += f()
    assert len({c.name for c in cases}) == len(cases)
    return cases


@functools.lru_cache(maxsize=None)
def cases() -> list[SCase]:
    return all_cases()


def test_every_case_fires_its_edge(oracle_mod):
    """Each case's edge fires on the oracle, and every planted ADV_EXT_IND is a CRC-ok record of the legacy decoder (so the
    engine's own poll provides the same sources)."""
    for c in cases():
        aux, got = c.lists()
        assert len(aux) and (aux["status"] == ao.OK).any(), c.name
        c.check(got)
        for cap_i, ch, s in c.spots:
            b = np.unpackbits(c.words[cap_i, ch, 4:].view(np.uint8), bitorder="little")[: c.n_out]
            rec = oracle_mod.ble_decode(bb.bits_to_iq(b), ch)
            pre, w0, _ = c.shard or (0, 0, 0)
            assert ((rec["sample_index"] == s - (8192 * w0 - pre)) & (rec["crc_ok"] == 1)).any(), (c.name, ch, s)


# ------------------------------------------------------------------------------------------------ end to end (CPU)
def end_to_end(oracle_mod, cap, taps_name: str):
    """numpy capture -> the channelizer's definition (pfb_oracle) -> quantiser and slicer -> the BLE oracle on 37..39 ->
    aux_oracle -> periodic_oracle (test_ble_aux.end_to_end, one step further)."""
    from test_ble_aux import _taps
    from snout_b200 import chanplan
    y = oracle_mod.pfb(cap.iq, _taps(taps_name), [chanplan.ble_channel_bin(c) for c in range(40)], fast=True)
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
    words = np.stack([bb.pack_words(b[c], n_words=4 + (n + 31) // 32 + 64) for c in range(40)])[None]
    aux = ao.aux_list(words, np.concatenate(frames), n)
    return aux, po.sync_list(words, aux, n)


def recovered(sync, truth, capture_id=0) -> int:
    got = {(int(r["channel"]), int(r["capture_id"]), bytes(r["bytes"][: int(r["len"])]))
           for r in sync if r["status"] == po.OK and r["crc_ok"]}
    return sum((t.channel, capture_id, t.data) in got for t in truth)


def test_end_to_end_recall(oracle_mod):
    cap = synth.periodic_adv_capture(seconds=0.05, seed=9710, esn0_db=25.0, n_trains=2, intervals=(6, 12))
    truth = [t for t in cap.meta["sync"] if not t.clash]
    assert len(truth) >= 6 and {t.phy for t in truth} == {0, 1}
    aux, sync = end_to_end(oracle_mod, cap, "BLE_384")
    assert recovered(sync, truth) == len(truth), (recovered(sync, truth), len(truth))
    assert (sync["event"] < 0).any()                     # events before the first AUX_ADV_IND are predicted backwards


# ------------------------------------------------------------------------------------------------ host side
def _sync_of_case():
    c = next(x for x in cases() if x.name == "equal_sources_two_trains")
    aux, sync = c.lists()
    return aux.astype(_abi.AUX_DTYPE), sync.astype(_abi.SYNC_DTYPE)


def test_periodic_messages():
    tr = Train(pa=3)
    s = 40_000
    sc = Scene(s + 4 * (15510 + 2 * 7500) + 4000, seed=11)
    sc.source(tr, s)
    big = bytes([34, 0x2C]) + bytes(33)
    p0 = sc.event(tr, s, 0, tr.window(0)[0] + 10, n=25, acad=big)
    p1 = sc.event(tr, s, 1, tr.window(1)[0] + 10, n=5, chained=True, crc_ok=False)
    c = case("msg", sc, lambda got: None)
    aux, sync = c.lists()
    (t,) = messages.ble_periodic_adv(sync.astype(_abi.SYNC_DTYPE), aux.astype(_abi.AUX_DTYPE))
    assert t["access_addr"] == tr.aa and t["crc_init"] == tr.crc_init and t["interval"] == 6 and t["interval_ms"] == 7.5
    assert t["channels"] == list(range(37)) and t["ppm"] == 500 and t["phy"] == "1M"
    assert t["adv_a"] == "060504030201" and t["adi"] == 0x1234
    e0, e1 = t["events"]
    assert e0["event"] == 0 and e0["event_counter"] == 3 and e0["crc_ok"] and e0["big_info"] and e0["acad"] == big
    assert e0["adv_data"] == p0[3 + (p0[2] & 0x3F):] and not e0["chained"]
    assert e1["chained"] and not e1["crc_ok"] and not e1["big_info"] and e1["acad"] == b""
    (t2,) = messages.ble_periodic_adv(sync.astype(_abi.SYNC_DTYPE))
    assert t2["adv_a"] is None and len(t2["events"]) == 2
    line = formats.sync_line(t, e0)
    assert line == f"SYNC Ch{tr.channel(0)} PHY1M AA:{tr.aa:08x} Evt3 Int6 PloadL{p0[1]} CRC0\n" and len(line.split()) == 8


def test_pcap_sync_block_bytes():
    aux, sync = _sync_of_case()
    blob = formats.ble_pcap_sync_block(sync)
    at, recs = 0, []
    while at < len(blob):
        n = struct.unpack(">i", blob[at + 8:at + 12])[0]
        recs.append(blob[at + 16:at + 16 + n])
        at += 16 + n
    ok = sync[sync["status"] == po.OK]
    assert len(recs) == len(ok) == 4
    for r, rec in zip(ok, recs):
        flags = struct.unpack("<H", rec[8:10])[0]
        assert rec[0] == r["channel"] and rec[1:8] == b"\0" * 7 and flags == 0x0001 | (1 << 7) | (int(r["phy"]) << 14)
        assert struct.unpack("<I", rec[10:14])[0] == r["access_addr"] and rec[14:] == bytes(r["bytes"][: int(r["len"]) - 3])


class SyncEngine(RecordingEngine):
    sync = None

    def ble_periodic(self):
        return self.sync


def test_cli_periodic(tmp_path):
    aux, sync = _sync_of_case()
    out = io.StringIO()
    assert btle_cli.run(btle_cli.parse_commandline(["--periodic", "--iq", "-"], out=out), out=out) == 1
    assert "--periodic needs --wideband" in out.getvalue()
    pcap = tmp_path / "x.pcap"
    SyncEngine.sync = sync
    out = io.StringIO()
    o = btle_cli.parse_commandline(["--wideband", "--periodic", "-s", str(pcap)], out=out)
    rc = btle_cli.run(o, out=out, engine_factory=lambda mode, **kw: SyncEngine(mode, **{k: v for k, v in kw.items() if k == "max_samples"}),
                      blocks=[np.zeros(24 * 8192, np.complex64)])
    assert rc == 0
    lines = [ln for ln in out.getvalue().splitlines() if ln.startswith("SYNC ")]
    assert len(lines) == 4 and all(len(ln.split()) == 8 for ln in lines)
    trains = messages.ble_periodic_adv(sync)
    assert lines[0] == formats.sync_line(trains[0], trains[0]["events"][0]).strip()
    data = pcap.read_bytes()
    assert data.startswith(formats.PCAP_HDR_BLE) and data.endswith(formats.ble_pcap_sync_block(sync))
