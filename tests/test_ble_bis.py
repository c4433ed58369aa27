"""BLE broadcast isochronous streams (snrx_ble_bis): the contract's restatement (oracle/bis_oracle.py) against the kernels'
host-side cores (tests/emu/emu_bis.cu) and synth's separate statement, constructed bit streams that put each edge of the
contract on the oracle, end to end through the channelizer's CPU statement, and the host side (messages, lines, pcap, CLI).
No GPU."""
from __future__ import annotations

import ctypes
import functools
import io
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

import ble_bits as bb
from fake_engine import RecordingEngine
from oracle import aux_oracle as ao
from oracle import bis_oracle as bo
from oracle import periodic_oracle as po
from snout_b200 import _abi, btle_cli, formats, messages, synth
from test_ble_periodic import KAT_NINE, Scene, Train, case, ext_header_sweep
from test_ble_periodic import _unmapped as unmapped_channel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bis_emu(tmp_path_factory):
    """tests/emu/emu_bis.cu (the cores of snout_b200/csrc/ble_bis.cuh) built with the flags of tests/emu/Makefile into a
    temporary directory."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = str(tmp_path_factory.mktemp("emu_bis") / "libemu_bis.so")
    r = subprocess.run([nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr",
                        "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-o", out,
                        os.path.join(ROOT, "tests", "emu", "emu_bis.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = ctypes.CDLL(out)
    lib.emu_bis_access_address.restype = ctypes.c_uint32
    lib.emu_bis_crc_init.restype = ctypes.c_uint32
    lib.emu_bis_channel.restype = ctypes.c_int
    lib.emu_bis_payload_number.restype = ctypes.c_uint64
    lib.emu_big_s_min.restype = ctypes.c_int64
    return lib


def _chm(used) -> int:
    return sum(1 << c for c in used)


def big_bytes(offset=100, units=30, iso=6, nb=2, nse=2, bn=1, sub=1000, pto=0, spacing=2000, irc=2, max_pdu=40, saa=0x3A1B5C2D,
              base=0xBEEF, used=range(37), phy=0, pc=1000, framing=0, enc=False) -> bytes:
    giv, gskd = (bytes(range(8)), bytes(range(16))) if enc else (None, None)
    return synth.big_info_bytes(offset, units, iso, nb, nse, bn, sub, pto, spacing, irc, max_pdu, saa, 10000, 40, base, _chm(used), phy,
                                pc, framing, giv, gskd)


def _buf(b: bytes):
    a = np.frombuffer(bytes(b), np.uint8).copy()
    return a, a.ctypes.data_as(ctypes.c_void_p)


# ------------------------------------------------------------------------------------------------ subevent channels
@pytest.mark.parametrize("aa,used,nse", [(0x8E89BED6, KAT_NINE, 4), (0x5A3C9E71, [0, 36], 3), (0x12345678, list(range(37)), 3),
                                         (0x0000FFFF, [5, 17, 18, 30], 2)])
def test_subevent_channels_kernel_equals_oracle_and_synth(bis_emu, aa, used, nse):
    chm = ctypes.c_uint64(_chm(used))
    n = len(used)
    d = max(1, min(3, n - 5), min(11, (n - 10) // 2))
    for c in range(65536):
        want = bo.subevent_channels(c, aa, used, nse)
        got = [bis_emu.emu_bis_channel(ctypes.c_uint32(c), ctypes.c_uint32(aa), chm, se) for se in range(nse)]
        assert got == want, c
        assert want[0] == po.csa2(c, aa, used)
        for a, b in zip(want, want[1:]):                     # consecutive subevents at least d apart in the used list
            gap = (used.index(b) - used.index(a)) % n
            assert d <= gap or n < 2 * d, (c, want)
        if c % 97 == 0:
            assert synth.csa2_subevent_channels(c, aa, used, nse) == want
    # long events on a few counters
    for c in (0, 1, 65535, 4000):
        want = bo.subevent_channels(c, aa, used, 31)
        assert [bis_emu.emu_bis_channel(ctypes.c_uint32(c), ctypes.c_uint32(aa), chm, se) for se in range(31)] == want
        assert synth.csa2_subevent_channels(c, aa, used, 31) == want


# ------------------------------------------------------------------------------------------------ access addresses, CRC init
def test_access_address_diversifier(bis_emu):
    rng = np.random.default_rng(31)
    for saa in [0, 0xFFFFFFFF] + [int(x) for x in rng.integers(0, 1 << 32, 1000, dtype=np.uint64)]:
        for n in range(32):
            want = bo.access_address(saa, n)
            assert bis_emu.emu_bis_access_address(ctypes.c_uint32(saa), n) == want == synth.bis_access_address(saa, n)
            assert (want ^ saa) & 0xFFFF == 0
    # the diversifier word, bit by bit: D = 42 for n = 0 (0101010), 77 for n = 1 (1001101)
    assert bo.access_address(0, 0) == 0b0000001010100100 << 16        # D0 = 0, D1 = 1, D6 = 0, D5 = 1, D4 = 0, D3 = 1, D2 = 0
    assert bo.access_address(0, 1) == 0b1111110100000110 << 16        # D0 = 1, D1 = 0, D6 = 1, D5 = 0, D4 = 0, D3 = 1, D2 = 1


def test_crc_init_convention(bis_emu):
    for base, n in ((0xBEEF, 1), (0x1234, 31), (0, 7), (0xFFFF, 2)):
        want = n << 16 | (base & 0xFF) << 8 | base >> 8
        assert bo.crc_init(base, n) == want == bis_emu.emu_bis_crc_init(ctypes.c_uint32(base), n)
        # the CRC seed of that crc_init is the 24-bit CRCInit base << 8 | n (sent least significant byte first)
        assert synth.sync_crc_seed(want) == synth.bis_crc_seed(base, n) == (base << 8 | n)


# ------------------------------------------------------------------------------------------------ BIGInfo parsing
FIELDS = ("offset", "units_us", "iso_interval", "num_bis", "nse", "bn", "sub_interval", "pto", "bis_spacing", "irc", "max_pdu",
          "sdu_interval", "max_sdu", "phy", "framing", "encrypted", "saa", "base_crc")


def _emu_find(bis_emu, pdu):
    f = (ctypes.c_int64 * 19)()
    chm, pc = ctypes.c_uint64(), ctypes.c_uint64()
    _, ptr = buf = _buf(pdu)
    rc = bis_emu.emu_big_info_find(ptr, pdu[1], f, ctypes.byref(chm), ctypes.byref(pc))
    del buf
    return None if rc < 0 else (list(f), chm.value, pc.value)


def _pdu_with(acad: bytes, **kw) -> bytes:
    return synth.ext_pdu(synth.ext_header(0, kw.get("adv_a"), 0, kw.get("adi"), None, kw.get("tx_power"), acad=acad), b"xy")


def test_big_info_fields_at_min_and_max(bis_emu):
    lo = dict(offset=0, units=30, iso=0, nb=0, nse=0, bn=0, sub=0, pto=0, spacing=0, irc=0, max_pdu=0, saa=0, base=0, used=[], phy=0, pc=0, framing=0)
    hi = dict(offset=16383, units=300, iso=4095, nb=31, nse=31, bn=7, sub=(1 << 20) - 1, pto=15, spacing=(1 << 20) - 1, irc=15, max_pdu=255,
              saa=0xFFFFFFFF, base=0xFFFF, used=range(37), phy=7, pc=(1 << 39) - 1, framing=1)
    for enc in (False, True):
        for v in (lo, hi):
            b = big_bytes(enc=enc, **v)
            assert len(b) == (57 if enc else 33)
            bi = bo.BigInfo(b)
            want = [v["offset"], v["units"], v["iso"], v["nb"], v["nse"], v["bn"], v["sub"], v["pto"], v["spacing"], v["irc"], v["max_pdu"],
                    10000, 40, v["phy"], v["framing"], int(enc), v["saa"], v["base"]]
            assert [int(getattr(bi, k)) for k in FIELDS] == want
            assert bi.chm == _chm(v["used"]) and bi.payload_count == v["pc"]
            pdu = _pdu_with(bytes([len(b) + 1, 0x2C]) + b)
            got = _emu_find(bis_emu, pdu)
            assert got is not None and got[0][:18] == [ctypes.c_int64(x).value for x in want] and got[1] == bi.chm and got[2] == bi.payload_count
            assert got[0][18] == int(bi.valid()) == 0                         # neither extreme is a valid BIG
            d = messages.big_info_fields(b)
            assert d["num_bis"] == v["nb"] and d["payload_count"] == v["pc"] and d["encrypted"] == enc and d["base_crc_init"] == v["base"]
    # other lengths are refused
    b = big_bytes()
    for ln in (32, 35, 57, 59):
        acad = bytes([ln, 0x2C]) + (b + bytes(64))[: ln - 1]
        assert bo.find_big_info(_pdu_with(acad), _pdu_with(acad)[1]) is None and _emu_find(bis_emu, _pdu_with(acad)) is None


def test_acad_walk(bis_emu):
    b = big_bytes()
    big = bytes([34, 0x2C]) + b
    cases = [
        (big, True),                                                   # first
        (bytes([3, 0xFF, 1, 2]) + big, True),                          # behind another AD structure
        (bytes([0]) + big, False),                                     # behind a length-0 structure: the walk stops
        (bytes([40, 0xFF]) + big, False),                              # behind one that overruns the ACAD
        (bytes([5, 0x2C, 1, 2, 3, 4]) + big, False),                   # the first 0x2C has the wrong length
        (bytes([3, 0xFF, 1, 2]), False),
    ]
    for acad, want in cases:
        for kw in ({}, dict(adv_a=b"\1" * 6, adi=0x1234, tx_power=-4)):
            pdu = _pdu_with(acad, **kw)
            got = bo.find_big_info(pdu, pdu[1])
            assert (got is not None) == want and (_emu_find(bis_emu, pdu) is not None) == want, (acad[:6], kw)
            if want:
                assert got.saa == 0x3A1B5C2D and got.valid()
    # a SyncInfo in front of the ACAD is skipped (18 bytes)
    si = synth.sync_info_bytes(100, 30, 6, 3, 0, 1, 2, 3)
    pdu = synth.ext_pdu(synth.ext_header(0, None, 0, None, None, None, sync_info=si, acad=big))
    assert bo.find_big_info(pdu, pdu[1]).saa == 0x3A1B5C2D and _emu_find(bis_emu, pdu) is not None


def test_big_info_find_on_every_header(bis_emu):
    """The kernels' ACAD walk equals the oracle's on every flags byte and header length, with a 0x2C structure (length 34, 58
    or random; a valid BIGInfo or random bytes) first in the ACAD or behind another structure."""
    rng = np.random.default_rng(20262)
    valid = (big_bytes(), big_bytes(enc=True))
    f, chm, pc = (ctypes.c_int64 * 19)(), ctypes.c_uint64(), ctypes.c_uint64()
    found = [0, 0]
    for buf, n_payload, flags, hlen in ext_header_sweep(20263):
        later = (flags + hlen + n_payload) % 2
        at = 2 + sum(size for bit, size in ((0, 6), (1, 6), (2, 1), (3, 2), (4, 3), (5, 18), (6, 1)) if flags >> bit & 1)
        ln = int(rng.choice([34, 58, rng.integers(1, 64)]))
        value = valid[ln == 58] if rng.integers(0, 2) else rng.integers(0, 256, 57, dtype=np.uint8).tobytes()
        ad = bytes([ln, 0x2C]) + value
        if later:
            m = int(rng.integers(1, 9))
            ad = bytes([m, 0xFF]) + rng.integers(0, 256, m - 1, dtype=np.uint8).tobytes() + ad
        ad = ad[: max(0, len(buf) - 2 - at)]
        buf[2 + at: 2 + at + len(ad)] = np.frombuffer(ad, np.uint8)
        want = bo.find_big_info(buf.tobytes(), n_payload)
        rc = bis_emu.emu_big_info_find(buf.ctypes.data_as(ctypes.c_void_p), n_payload, f, ctypes.byref(chm), ctypes.byref(pc))
        assert (rc == 0) == (want is not None), (flags, hlen, n_payload, later)
        if want is not None:
            assert list(f) == [int(getattr(want, k)) for k in FIELDS] + [int(want.valid())], (flags, hlen, n_payload, later)
            assert chm.value == want.chm and pc.value == want.payload_count, (flags, hlen, n_payload, later)
            found[later] += 1
    assert min(found) > 100                                        # hits at the first and at a later position


def test_validity_rules():
    assert bo.BigInfo(big_bytes()).valid()
    bad = [dict(nb=0), dict(bn=0), dict(nse=0), dict(nse=3, bn=2), dict(irc=0), dict(nse=4, bn=2, irc=3), dict(iso=3), dict(phy=2),
           dict(used=[4]), dict(spacing=7500 - 1000 + 1, nb=2, nse=2, sub=1000), dict(nse=2, sub=0), dict(nse=2, sub=7500, spacing=0)]
    for kw in bad:
        assert not bo.BigInfo(big_bytes(**kw)).valid(), kw
    good = [dict(iso=4, nb=1, nse=1, sub=0, spacing=0, irc=1), dict(phy=1), dict(used=[4, 5]), dict(nse=4, bn=2, irc=2, pto=3)]
    for kw in good:
        assert bo.BigInfo(big_bytes(**kw)).valid(), kw


# ------------------------------------------------------------------------------------------------ payload numbers
def test_payload_numbers(bis_emu):
    rng = np.random.default_rng(7)
    checked = 0
    for nse in range(1, 32):
        for bn in range(1, 8):
            if nse % bn:
                continue
            for irc in range(1, min(nse // bn, 15) + 1):         # IRC has 4 bits
                for pto in (0, 1, 15):
                    pc = int(rng.integers(0, 1 << 39))
                    b = big_bytes(nse=nse, bn=bn, irc=irc, pto=pto, pc=pc)
                    a, ptr = _buf(b)
                    bi = bo.BigInfo(b)
                    for k in (-3, 0, 5):
                        for se in range(nse):
                            want = bo.payload_number(bi, k, se)
                            assert bis_emu.emu_bis_payload_number(ptr, 33, ctypes.c_int64(k), se) == want
                            assert synth.bis_payload_number(pc, bn, irc, pto, k, se) == want
                            checked += 1
    assert checked > 10000
    # a pretransmission group: NSE 4, BN 2, IRC 1, PTO 2 -- subevents 2, 3 carry event k + 2's payloads
    bi = bo.BigInfo(big_bytes(nse=4, bn=2, irc=1, pto=2, pc=20))
    assert [bo.payload_number(bi, 0, se) for se in range(4)] == [20, 21, 24, 25]
    # the 39-bit wrap, forwards and backwards
    bi = bo.BigInfo(big_bytes(nse=2, bn=1, irc=1, pto=1, pc=(1 << 39) - 1))
    assert bo.payload_number(bi, 0, 1) == 0 and bo.BigInfo(big_bytes(pc=0)).payload_count == 0
    assert bo.payload_number(bo.BigInfo(big_bytes(pc=0, irc=2)), -1, 0) == (1 << 39) - 1


# ------------------------------------------------------------------------------------------------ windows and listed events
def _emu_window(bis_emu, b, ppm, k, n, se):
    a, ptr = _buf(b)
    lo, hi = ctypes.c_int64(), ctypes.c_int64()
    bis_emu.emu_bis_window(ptr, len(b), ppm, ctypes.c_int64(k), n, se, ctypes.byref(lo), ctypes.byref(hi))
    return lo.value, hi.value


def _emu_range(bis_emu, b, ppm, s, sps, base, n_out):
    a, ptr = _buf(b)
    x, y = ctypes.c_int64(), ctypes.c_int64()
    bis_emu.emu_big_k_range(ptr, len(b), ppm, ctypes.c_int64(s), sps, ctypes.c_int64(base), ctypes.c_int64(n_out), ctypes.byref(x), ctypes.byref(y))
    return x.value, y.value


def random_big(rng, phy=None) -> bytes:
    """A random valid BIGInfo, sequential or interleaved."""
    while True:
        iso = int(rng.choice([4, 5, 6, 8, 16, 80, 400]))
        nb, bn = int(rng.integers(1, 6)), int(rng.integers(1, 4))
        nse = bn * int(rng.integers(1, 5))
        irc = int(rng.integers(1, nse // bn + 1))
        I = 1250 * iso
        if rng.integers(0, 2):
            sub = int(rng.integers(150, max(151, I // (nse + 1))))
            spacing = int(rng.integers(nse * sub, nse * sub + 200)) if nb > 1 else 0
        else:
            spacing = int(rng.integers(150, max(151, I // (nb * nse + 1))))
            sub = nb * spacing
        b = big_bytes(offset=int(rng.integers(0, 16384)), units=int(rng.choice([30, 300])), iso=iso, nb=nb, nse=nse, bn=bn, sub=sub,
                      spacing=spacing, irc=irc, pto=int(rng.integers(0, 4)), phy=int(rng.integers(0, 2)) if phy is None else phy,
                      pc=int(rng.integers(0, 1 << 39)))
        if bo.BigInfo(b).valid():
            return b


def test_kernel_window_and_range_equal_the_oracle(bis_emu):
    rng = np.random.default_rng(5)
    n_nonempty = 0
    for i in range(150):
        b = random_big(rng)
        bi = bo.BigInfo(b)
        ppm = po.SCA_PPM[int(rng.integers(0, 8))] if i % 3 else 500
        for k in rng.integers(-300, 300, 3):
            for n, se in ((1, 0), (bi.num_bis, bi.nse - 1), (int(rng.integers(1, bi.num_bis + 1)), int(rng.integers(0, bi.nse)))):
                assert _emu_window(bis_emu, b, ppm, int(k), n, se) == bo.window(bi, ppm, int(k), n, se)
        sps = bi.sps
        s = int(rng.integers(0, 4_000_000))
        base = int(rng.integers(-2_000_000, s + 1))
        n_out = int(rng.integers(2, 6_000_000))
        r = bo.listed_range(bi, ppm, s, base, n_out)
        got = _emu_range(bis_emu, b, ppm, s, sps, base, n_out)
        if len(r):
            n_nonempty += 1
            assert got == (r.start, r.stop - 1), (got, r)
        else:
            assert got[1] < got[0]
    assert n_nonempty > 30
    # negative D, at a known point: O = 3000, I' = 7500, k = -1, first subevent: D = -4500
    bi = bo.BigInfo(big_bytes())
    assert bo.window(bi, 500, -1, 1, 0) == ((4 * -4500 * 1000500) // 10**6 - 8, -((-4 * -4470 * 999500) // 10**6) + 8)
    assert _emu_window(bis_emu, big_bytes(), 500, -1, 1, 0) == bo.window(bi, 500, -1, 1, 0)


@pytest.mark.parametrize("kw,ppm", [(dict(), 500), (dict(nse=1, sub=0, irc=1, iso=4, spacing=1500), 500),
                                    (dict(nse=3, sub=2400, spacing=7300, nb=1, irc=3), 500),      # S_min = 7500 - 2 sub = 2700 > sub: sub
                                    (dict(nse=3, sub=3000, spacing=0, nb=1, irc=3), 500),         # S_min = 7500 - 6000 = 1500 < sub
                                    (dict(nb=3, spacing=400, sub=1200, nse=2, irc=2), 150)])      # interleaved
def test_rule_a_last_listed_and_first_unlisted(bis_emu, kw, ppm):
    b = big_bytes(**kw)
    bi = bo.BigInfo(b)
    smin = bi.s_min
    assert bis_emu.emu_big_s_min(_buf(b)[1], 33) == smin
    r = bo.listed_range(bi, ppm, 10**12, 0, 2 * 10**12)
    assert len(r) > 2
    for k, inside in ((r.start, True), (r.start - 1, False), (r.stop - 1, True), (r.stop, False)):
        assert bo.event_ok(bi, ppm, k) == inside
    assert _emu_range(bis_emu, b, ppm, 10**12, bi.sps, 0, 2 * 10**12) == (r.start, r.stop - 1)


@pytest.mark.parametrize("sub,k", [(481, 27), (1473, 93)])
def test_rule_a_at_exactly_half_the_spacing(bis_emu, sub, k):
    """A window of exactly 2 S_min samples is listed (rule (a) is <=), the next event's is not."""
    b = big_bytes(nse=2, nb=1, spacing=0, sub=sub, irc=2)
    bi = bo.BigInfo(b)
    widths = [bo.window(bi, 500, k, 1, se)[1] - bo.window(bi, 500, k, 1, se)[0] + 1 for se in range(2)]
    assert max(widths) == 2 * bi.s_min
    r = bo.listed_range(bi, 500, 10**12, 0, 2 * 10**12)
    assert r.stop - 1 == k
    assert _emu_range(bis_emu, b, 500, 10**12, 4, 0, 2 * 10**12) == (r.start, k)


def test_windows_of_a_bis_are_disjoint():
    """The contract's bound, swept over random valid BIGInfos: every window of a listed event is at most 2 S_min samples, so
    with the 31 sps address span it ends before the next window of its BIS starts."""
    rng = np.random.default_rng(2025)
    for i in range(20000):
        b = random_big(rng)
        bi = bo.BigInfo(b)
        ppm = po.SCA_PPM[i % 8]
        kc = bo.k_c(bi)
        for k in (kc - 2, kc - 1, kc, kc + 1):
            if not bo.event_ok(bi, ppm, k):
                continue
            for n in range(1, bi.num_bis + 1):
                wins = [bo.window(bi, ppm, k, n, se) for se in range(bi.nse)]
                if bo.event_ok(bi, ppm, k + 1):
                    wins.append(bo.window(bi, ppm, k + 1, n, 0))
                for (lo0, hi0), (lo1, hi1) in zip(wins, wins[1:]):
                    assert hi0 + 31 * bi.sps < lo1, (i, k, n)


def test_windows_of_a_bis_are_disjoint_at_the_rule_a_edges(bis_emu):
    """The same bound where it binds: at the first and last events of rule (a)'s range, whose windows come close to 2 S_min
    samples.  The range's edges come from the kernels' k range on a buffer too long for rule (b) to cut it (equal to the
    oracle's brute-force range in test_kernel_window_and_range_equal_the_oracle); the oracle confirms both are edges."""
    rng = np.random.default_rng(2026)
    widest = 0.0
    for i in range(3000):
        b = random_big(rng)
        bi = bo.BigInfo(b)
        ppm = po.SCA_PPM[i % 8]
        a, z = _emu_range(bis_emu, b, ppm, 10**12, bi.sps, 0, 2 * 10**12)
        if z < a:
            continue
        assert bo.event_ok(bi, ppm, a) and bo.event_ok(bi, ppm, z)
        assert not bo.event_ok(bi, ppm, a - 1) and not bo.event_ok(bi, ppm, z + 1)
        for k0, k1 in ((a, a + 1), (z - 1, z)):
            if k1 > z or k0 < a:
                continue
            for n in range(1, bi.num_bis + 1):
                wins = [bo.window(bi, ppm, k0, n, se) for se in range(bi.nse)] + [bo.window(bi, ppm, k1, n, se) for se in range(bi.nse)]
                for (lo0, hi0), (lo1, hi1) in zip(wins, wins[1:]):
                    assert hi0 + 31 * bi.sps < lo1, (i, k0, n)
                widest = max(widest, max(hi - lo + 1 for lo, hi in wins) / (2 * bi.s_min))
    assert widest > 0.99                                         # the edges reach windows of about 2 S_min


# ------------------------------------------------------------------------------------------------ constructed streams
class Big:
    """A BIG's BIGInfo and the symbols of its BIS PDUs, predicted from a carrier at sample c (train ppm `ppm`)."""

    def __init__(self, ppm=500, **kw):
        self.bytes = big_bytes(**kw)
        self.bi = bo.BigInfo(self.bytes)
        self.ppm = ppm
        self.sps = self.bi.sps

    def acad(self) -> bytes:
        return bytes([len(self.bytes) + 1, 0x2C]) + self.bytes

    def aa(self, n):
        return bo.access_address(self.bi.saa, n)

    def counter(self, k):
        return (self.bi.payload_count // self.bi.bn + k) % 65536

    def window(self, k, n, se):
        return bo.window(self.bi, self.ppm, k, n, se)

    def channel(self, k, n, se):
        return bo.subevent_channels(self.counter(k), self.aa(n), self.bi.used, self.bi.nse)[se]


def bis_pdu(rng, n=12) -> bytes:
    return bytes([0x02 | (3 << 2), n]) + bytes(rng.integers(0, 256, n, dtype=np.uint8))


class BScene(Scene):
    def carrier(self, tr: Train, s: int, big: Big, k: int = 0, at: int = 10, extra_acad: bytes = b"") -> int:
        """The train's source at s and its event k at win_lo + at, carrying big's BIGInfo; returns the carrier's sample."""
        if not any(np.any(f["sample_index"] == s - 2400) for f in self.bt.frames):
            self.source(tr, s)
        c = s + tr.window(k)[0] + at
        self.event(tr, s, k, tr.window(k)[0] + at, n=4, acad=extra_acad + big.acad())
        return c

    def bis(self, big: Big, c: int, k: int, n: int, se: int, at: int, ln: int = 12, crc_ok=True) -> bytes:
        """The BIS PDU of subevent (n, se) of event k, AA bit 0 at c + at."""
        pdu = bis_pdu(self.rng, ln)
        sym = bb.frame_symbols(big.channel(k, n, se), pdu[:2], pdu[2:], crc_ok, aa=big.aa(n), crc_init=synth.bis_crc_seed(big.bi.base_crc, n))
        from test_ble_aux import plant_stride
        plant_stride(self.bt.b[big.channel(k, n, se)], c + at, sym, big.sps)
        return pdu


def lists(c):
    aux, sync = c.lists()
    return aux, sync, bo.bis_list(c.words, sync, c.n_out, **c.geo())


def ent(got, k, n, se, source=None):
    sel = (got["event"] == k) & (got["bis"] == n) & (got["subevent"] == se)
    if source is not None:
        sel &= got["source"] == source
    (r,) = got[sel]
    return r


def found(r, big: Big, at: int, pdu: bytes, k: int, n: int, se: int):
    want = pdu + synth.ble_crc24(pdu, synth.bis_crc_seed(big.bi.base_crc, n))
    assert r["status"] == bo.OK and int(r["sample_index"]) == at and r["channel"] == big.channel(k, n, se)
    assert r["len"] == len(want) and r["crc_ok"] and bytes(r["bytes"][: len(want)]) == want
    assert r["access_addr"] == big.aa(n) and r["crc_init"] == bo.crc_init(big.bi.base_crc, n) and r["event_counter"] == big.counter(k)
    assert r["payload_number"] == bo.payload_number(big.bi, k, se)


S0 = 60_000                       # the train's source
TR = dict(offset=517, sca=0)      # carrier at S0 + window(0)[0] + 10 = S0 + 62 022


def _window_edges():
    out = []
    tr = Train(**TR)
    for k in (-2, 1):
        for n, se in ((1, 0), (2, 1)):
            for name, d, hit in (("lo-1", -1, False), ("lo", 0, True), ("hi", 0, True), ("hi+1", 1, False)):
                big = Big()
                sc = BScene(S0 + 140_000, seed=abs(k) * 100 + n * 10 + len(name))
                c = sc.carrier(tr, S0, big)
                lo, hi = big.window(k, n, se)
                at = (lo if name.startswith("lo") else hi) + d
                pdu = sc.bis(big, c, k, n, se, at)

                def check(got, k=k, n=n, se=se, at=at, hit=hit, pdu=pdu, big=big, c=c):
                    r = ent(got, k, n, se)
                    assert (int(r["win_lo"]), int(r["win_hi"])) == (c + big.window(k, n, se)[0], c + big.window(k, n, se)[1])
                    if hit:
                        found(r, big, c + at, pdu, k, n, se)
                    else:
                        assert r["status"] == bo.NOT_FOUND and r["sample_index"] == -1
                out.append(case(f"edge_k{k}_{n}{se}_{name}", sc, check))
    return out


def _buffer_ends():
    """OUTSIDE at both ends, the first and last listed events, TRUNCATED / OK at the end."""
    out = []
    tr = Train(**TR)
    for phy in (0, 1):
        big = Big(phy=phy)
        sps = big.sps
        c0 = S0 + tr.window(0)[0] + 10
        # the start: event -3's first window starts at sample d (the source is moved so; its primary stays in the buffer)
        lo = big.window(-3, 1, 0)[0]
        for d, want in ((0, "searched"), (-1, "outside")):
            shift = -(c0 + lo) + d
            assert S0 + shift - 2400 >= 500, "the source's primary must stay inside the buffer"
            sc = BScene(S0 + shift + 140_000, seed=5 + d + sps)
            c = sc.carrier(tr, S0 + shift, big)
            pdu = sc.bis(big, c, -3, 1, 0, lo + 5)

            def check(got, d=d, want=want, big=big, c=c, pdu=pdu, lo=lo):
                r = ent(got, -3, 1, 0)
                assert int(r["win_lo"]) == d and (r["status"] == bo.OUTSIDE) == (want == "outside")
                if want == "searched":
                    found(r, big, c + lo + 5, pdu, -3, 1, 0)
                assert got["event"].min() == -3                            # the first listed event
                assert c + big.window(-4, 2, 1)[1] + 31 * big.sps < 0      # event -4 misses the buffer
                assert (got[got["event"] == -3]["status"] != bo.OUTSIDE).sum() >= 3
            out.append(case(f"start_{sps}_{want}", sc, check))
        # the end: the last subevent of event 1 at the last usable decision
        c = c0
        hi = big.window(1, 2, 1)[1]
        lo1 = big.window(1, 1, 0)[0]
        for n_out, want in ((c + hi + 31 * sps + 2, "searched"), (c + hi + 31 * sps + 1, "outside"), (c + lo1 + 2, "lo_last"),
                            (c + lo1 + 1, "unlisted")):
            sc = BScene(n_out, seed=n_out % 1000)
            sc.carrier(tr, S0, big)

            def check(got, want=want, n_out=n_out, c=c, big=big):
                if want == "unlisted":
                    assert got["event"].max() == 0
                    return
                r = ent(got, 1, 2, 1)
                assert (r["status"] == bo.OUTSIDE) == (want in ("outside", "lo_last"))
                if want == "lo_last":
                    assert int(ent(got, 1, 1, 0)["win_lo"]) == n_out - 2
            out.append(case(f"end_{sps}_{want}", sc, check))
        # TRUNCATED at the end
        at = big.window(1, 2, 1)[1] - 4
        ln = 40
        end = c + at + (32 + 8 * (2 + ln + 3) - 1) * sps
        for n_out, status in ((end + 2, bo.OK), (end + 1, bo.TRUNCATED)):
            sc = BScene(n_out, seed=n_out % 997)
            sc.carrier(tr, S0, big)
            sc.bis(big, c, 1, 2, 1, at, ln=ln)

            def check(got, status=status, at=at, c=c):
                r = ent(got, 1, 2, 1)
                assert r["status"] == status and int(r["sample_index"]) == c + at
            out.append(case(f"trunc_{sps}_{n_out - end}", sc, check))
    return out


def _phases_wrap_remap_encrypted():
    out = []
    tr = Train(**TR)
    for phase in (0, 1):
        big = Big(phy=1, nb=3, nse=4, bn=2, irc=1, pto=1, sub=500, spacing=2000)
        sc = BScene(S0 + 140_000, seed=20 + phase)
        c = sc.carrier(tr, S0, big, at=10 + phase)
        pdus = {(k, n, se): sc.bis(big, c, k, n, se, big.window(k, n, se)[0] + 11 + phase) for k in (-1, 0, 1) for n, se in ((1, 0), (3, 3), (2, 2))}

        def check(got, big=big, c=c, pdus=pdus, phase=phase):
            for (k, n, se), pdu in pdus.items():
                r = ent(got, k, n, se)
                found(r, big, c + big.window(k, n, se)[0] + 11 + phase, pdu, k, n, se)
                assert r["phase"] == int(r["sample_index"]) % 2 and r["phy"] == ao.PHY_2M
            assert {int(ent(got, *key)["phase"]) for key in pdus} == {0, 1}
        out.append(case(f"2m_phase{phase}", sc, check))
    for pc in (65535, 65536 * 5):
        big = Big(pc=pc, used=KAT_NINE, saa=0x8E89BED7, nse=3, irc=3)
        sc = BScene(S0 + 140_000, seed=pc % 13)
        c = sc.carrier(tr, S0, big)
        ks = (0, 1) if pc == 65535 else (-1, 0)
        pdus = {(k, n, se): sc.bis(big, c, k, n, se, big.window(k, n, se)[0] + 9) for k in ks for n in (1, 2) for se in range(3)}

        def check(got, big=big, c=c, pdus=pdus):
            for (k, n, se), pdu in pdus.items():
                found(ent(got, k, n, se), big, c + big.window(k, n, se)[0] + 9, pdu, k, n, se)
            assert {0, 65535} <= {int(ent(got, k, 1, 0)["event_counter"]) for k, _, _ in pdus}
        out.append(case(f"wrap_{pc}", sc, check))
    # remapped channels: subevent 0 of events whose unmapped channel is not used, and later subevents
    big = Big(used=[2, 11, 29], saa=0x71764129, pc=4000, nse=2)
    sc = BScene(S0 + 140_000, seed=9)
    c = sc.carrier(tr, S0, big)
    pdus = {(k, n, se): sc.bis(big, c, k, n, se, big.window(k, n, se)[1] - 3) for k in (-1, 0, 1) for n in (1, 2) for se in (0, 1)}

    def check_remap(got, big=big, c=c):
        for (k, n, se), pdu in pdus.items():
            found(ent(got, k, n, se), big, c + big.window(k, n, se)[1] - 3, pdu, k, n, se)
        remapped = 0
        for k, n, _ in pdus:                                     # subevent 0 whose unmapped channel prn_e mod 37 is not used
            aa = big.aa(n)
            remapped += unmapped_channel(big.counter(k), ((aa >> 16) ^ aa) & 0xFFFF) not in big.bi.used
        assert remapped >= 2
    out.append(case("remap", sc, check_remap))
    # an encrypted BIGInfo (57 bytes), framed: the payload (with its MIC) as sent
    big = Big(enc=True, framing=1)
    sc = BScene(S0 + 140_000, seed=31)
    c = sc.carrier(tr, S0, big)
    pdu = sc.bis(big, c, 0, 2, 0, big.window(0, 2, 0)[0] + 40, ln=20)

    def check_enc(got, big=big, c=c, pdu=pdu):
        r = ent(got, 0, 2, 0)
        found(r, big, c + big.window(0, 2, 0)[0] + 40, pdu, 0, 2, 0)
        assert (got["flags"] == bo.ENCRYPTED | bo.FRAMED).all()
    out.append(case("encrypted", sc, check_enc))
    # an SAA whose AA_1 is 0: its entries are NOT_FOUND although 32 zero decisions sit in every window
    saa0 = bo.access_address(0, 1)
    big = Big(saa=saa0)
    assert big.aa(1) == 0 and big.aa(2) != 0
    sc = BScene(S0 + 140_000, seed=41)
    c = sc.carrier(tr, S0, big)
    for ch in range(37):
        lo, hi = big.window(0, 1, 0)
        sc.bt.b[ch][c + lo - 200:c + hi + 400] = 0
    pdu2 = sc.bis(big, c, 0, 2, 0, big.window(0, 2, 0)[0] + 5)

    def check_zero(got, big=big, c=c, pdu2=pdu2):
        assert (got[got["bis"] == 1]["status"] != bo.OK).all() and ent(got, 0, 1, 0)["status"] == bo.NOT_FOUND
        found(ent(got, 0, 2, 0), big, c + big.window(0, 2, 0)[0] + 5, pdu2, 0, 2, 0)
    out.append(case("aa_zero", sc, check_zero))
    return out


def _sources_and_bigs():
    out = []
    # two carriers of one SAA at the same sample (different channels and trains: the lower list index wins), a later one
    # with another offset, and a second BIG whose window is wider than two 32-word passes (U = 300 us)
    a_tr, b_tr, c_tr = Train(**TR), Train(aa=0x3F1E2D4C, crc_init=0xA5A5A5, **TR), Train(aa=0x21436587, crc_init=0x5A5A5A, **TR)
    big = Big(offset=100)
    big_late = Big(offset=90)
    wide = Big(saa=0x55AA33CC, base=0x1357, offset=20, units=300, nb=1, nse=2, irc=2, sub=3000, spacing=0)
    sc = BScene(S0 + 140_000, seed=3)
    c1 = sc.carrier(a_tr, S0, big)
    sc.source(b_tr, S0 + 4000, ch=6, prim_channel=38)
    c2 = S0 + 4000 + b_tr.window(0)[0] + 10
    sc.event(b_tr, S0 + 4000, 0, b_tr.window(0)[0] + 10, n=4, acad=big_late.acad())
    sc.source(c_tr, S0 + 9000, ch=8, prim_channel=39)
    c3 = S0 + 9000 + c_tr.window(0)[0] + 10
    sc.event(c_tr, S0 + 9000, 0, c_tr.window(0)[0] + 10, n=4, acad=wide.acad())
    pa = {(k, n): sc.bis(big, c1, k, n, 0, big.window(k, n, 0)[0] + 12) for k in (0, 1) for n in (1, 2)}
    lo, hi = wide.window(0, 1, 1)
    assert hi - lo > 1024 + 64
    pw = sc.bis(wide, c3, 0, 1, 1, hi - 2)

    def check(got, c1=c1, c3=c3):
        srcs = sorted(set(got["source"].tolist()))
        assert len(srcs) == 2
        ga, gw = got[got["source"] == srcs[0]], got[got["source"] == srcs[1]]
        for (k, n), pdu in pa.items():
            found(ent(ga, k, n, 0), big, c1 + big.window(k, n, 0)[0] + 12, pdu, k, n, 0)     # predicted from the first carrier
        found(ent(gw, 0, 1, 1), wide, c3 + hi - 2, pw, 0, 1, 1)
        assert got["source"].tolist() == sorted(got["source"].tolist())
    out.append(case("earlier_carrier_two_bigs", sc, check))
    assert c2 > c1
    # ties: two carriers of one SAA at the same sample on different channels; the lower list index is the source
    t1, t2 = Train(aa=0x11223344, **TR), Train(aa=0x55667788, crc_init=0x123456, **TR)
    sc = BScene(S0 + 140_000, seed=4)
    sc.source(t1, S0, ch=5, prim_channel=37)
    sc.source(t2, S0, ch=7, prim_channel=38)
    c = S0 + t1.window(0)[0] + 10
    b1, b2 = Big(offset=100), Big(offset=104)
    sc.event(t1, S0, 0, t1.window(0)[0] + 10, n=4, acad=b1.acad())
    sc.event(t2, S0, 0, t2.window(0)[0] + 10, n=4, acad=b2.acad())
    p = sc.bis(b1, c, 0, 1, 0, b1.window(0, 1, 0)[0] + 3)

    def check_tie(got, c=c, p=p):
        assert len(set(got["source"].tolist())) == 1
        r = ent(got, 0, 1, 0)
        found(r, b1, c + b1.window(0, 1, 0)[0] + 3, p, 0, 1, 0)
    out.append(case("tie_lower_index", sc, check_tie))
    return out


def _captures_and_shards():
    out = []
    tr = Train(**TR)
    big = Big()
    scenes, pdus = [], []
    for cap in range(3):
        sc = BScene(S0 + 140_000, seed=40 + cap)
        if cap != 1:
            c = sc.carrier(tr, S0 + 100 * cap, big)
            pdus.append((c, sc.bis(big, c, 1, 2, 1, big.window(1, 2, 1)[0] + 20 + cap)))
        scenes.append(sc)

    def check(got):
        assert sorted(set(got["capture_id"].tolist())) == [5, 7]
        for cap, (c, pdu) in zip((0, 2), pdus):
            g = got[got["capture_id"] == 5 + cap]
            found(ent(g, 1, 2, 1), big, c + big.window(1, 2, 1)[0] + 20 + cap, pdu, 1, 2, 1)
    out.append(case("three_captures", scenes, check, first_capture=5))
    w0, pre = 3, 128
    base = 8192 * w0 - pre
    s = base + S0
    whole = BScene(s + 140_000, seed=77)
    c = whole.carrier(tr, s, big)
    p = {k: whole.bis(big, c, k, 1, 1, big.window(k, 1, 1)[0] + 30) for k in (-1, 0, 1)}
    sh = BScene(whole.bt.n - base, seed=78)
    for ch in list(whole.bt.b):
        sh.bt.b[ch] = whole.bt.b[ch][base:].copy()
    sh.bt.frames = [f.copy() for f in whole.bt.frames]

    def check_shard(got, c=c):
        for k, pdu in p.items():
            found(ent(got, k, 1, 1), big, c + big.window(k, 1, 1)[0] + 30, pdu, k, 1, 1)
    out.append(case("shard", sh, check_shard, shard=(pre, w0, (sh.bt.n - pre) // 8192)))
    return out


def all_cases():
    cases_ = []
    for f in (_window_edges, _buffer_ends, _phases_wrap_remap_encrypted, _sources_and_bigs, _captures_and_shards):
        cases_ += f()
    assert len({c.name for c in cases_}) == len(cases_)
    return cases_


@functools.lru_cache(maxsize=None)
def cases():
    return all_cases()


def test_every_case_fires_its_edge():
    names = {c.name for c in cases()}
    for sps in (4, 2):                                           # both buffer ends are built, for both PHYs
        assert {f"start_{sps}_searched", f"start_{sps}_outside", f"end_{sps}_searched", f"end_{sps}_outside",
                f"end_{sps}_lo_last", f"end_{sps}_unlisted"} <= names
    for c in cases():
        aux, sync, got = lists(c)
        assert len(sync) and len(got), c.name
        c.check(got)


# ------------------------------------------------------------------------------------------------ end to end (CPU)
def recovered(bis, truth, capture_id=0) -> int:
    got = {(int(r["channel"]), int(r["capture_id"]), bytes(r["bytes"][: int(r["len"])]))
           for r in bis if r["status"] == bo.OK and r["crc_ok"]}
    return sum((t.channel, capture_id, t.data) in got for t in truth)


def end_to_end(oracle_mod, cap, taps_name: str = "BLE_384"):
    """numpy capture -> the channelizer's definition (pfb_oracle) -> quantiser and slicer -> the BLE oracle on 37..39 ->
    aux_oracle -> periodic_oracle -> bis_oracle (test_ble_periodic.end_to_end, one step further)."""
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
    sync = po.sync_list(words, aux, n)
    return sync, bo.bis_list(words, sync, n)


def test_end_to_end_recall(oracle_mod):
    cap = synth.broadcast_iso_capture(seconds=0.05, seed=9910, esn0_db=25.0)
    truth = [t for t in cap.meta["bis"] if not t.clash]
    assert len(truth) >= 40 and {t.phy for t in truth} == {0, 1}
    sync, bis = end_to_end(oracle_mod, cap)
    assert recovered(bis, truth) == len(truth), (recovered(bis, truth), len(truth))
    assert (bis["event"] < 0).any() and (bis["flags"] & bo.ENCRYPTED).any()


# ------------------------------------------------------------------------------------------------ host side
def _lists_of_case(name="earlier_carrier_two_bigs"):
    c = next(x for x in cases() if x.name == name)
    aux, sync, bis = lists(c)
    return sync.astype(_abi.SYNC_DTYPE), bis.astype(_abi.BIS_DTYPE)


def test_broadcast_iso_messages_and_lines():
    sync, bis = _lists_of_case()
    bigs = messages.ble_broadcast_iso(bis, sync)
    assert len(bigs) == 2
    g = bigs[0]
    assert g["big_info"]["num_bis"] == 2 and g["big_info"]["iso_interval_ms"] == 7.5 and g["phy"] == "1M"
    assert [s["bis"] for s in g["streams"]] == [1, 2]
    s1 = g["streams"][0]
    assert s1["access_addr"] == bo.access_address(0x3A1B5C2D, 1) and s1["crc_init"] == bo.crc_init(0xBEEF, 1)
    p = s1["pdus"][0]
    ok = bis[(bis["source"] == g["source"]) & (bis["bis"] == 1) & (bis["status"] == bo.OK)][0]
    pdu = bytes(ok["bytes"][: int(ok["len"])])
    assert p["llid"] == pdu[0] & 3 and p["cssn"] == (pdu[0] >> 2) & 7 and p["cstf"] == (pdu[0] >> 5) & 1
    assert p["payload"] == pdu[2:2 + pdu[1]] and p["pload_len"] == pdu[1] and p["crc_ok"] and not p["encrypted"]
    assert p["payload_number"] == int(ok["payload_number"]) and p["subevent"] == int(ok["subevent"])
    (g2, _) = messages.ble_broadcast_iso(bis)
    assert g2["big_info"] is None and len(g2["streams"]) == 2
    line = formats.bis_line(g, s1, p)
    assert line == (f"BIS Ch{int(ok['channel'])} PHY1M AA:{s1['access_addr']:08x} BIS1 Evt{int(ok['event_counter'])} Se{int(ok['subevent'])} "
                    f"PloadL{pdu[1]} CRC0\n") and len(line.split()) == 9


def test_pcap_bis_block_bytes():
    sync, bis = _lists_of_case()
    blob = formats.ble_pcap_bis_block(bis)
    at, recs = 0, []
    while at < len(blob):
        n = struct.unpack(">i", blob[at + 8:at + 12])[0]
        recs.append(blob[at + 16:at + 16 + n])
        at += 16 + n
    ok = bis[bis["status"] == bo.OK]
    assert len(recs) == len(ok) >= 5
    for r, rec in zip(ok, recs):
        flags = struct.unpack("<H", rec[8:10])[0]
        assert rec[0] == r["channel"] and rec[1:8] == b"\0" * 7
        assert flags == formats.PHDR_DEWHITENED | (formats.PHDR_PDU_BIS << formats.PHDR_PDU_TYPE_SHIFT) | (int(r["phy"]) << formats.PHDR_PHY_SHIFT)
        assert struct.unpack("<I", rec[10:14])[0] == r["access_addr"] and rec[14:] == bytes(r["bytes"][: int(r["len"]) - 3])


class BisEngine(RecordingEngine):
    bis = None

    def ble_bis(self):
        return self.bis


def test_cli_bis(tmp_path):
    sync, bis = _lists_of_case()
    out = io.StringIO()
    assert btle_cli.run(btle_cli.parse_commandline(["--bis", "--iq", "-"], out=out), out=out) == 1
    assert "--bis needs --wideband" in out.getvalue()
    pcap = tmp_path / "x.pcap"
    BisEngine.bis = bis
    out = io.StringIO()
    o = btle_cli.parse_commandline(["--wideband", "--bis", "-s", str(pcap)], out=out)
    rc = btle_cli.run(o, out=out, engine_factory=lambda mode, **kw: BisEngine(mode, **{k: v for k, v in kw.items() if k == "max_samples"}),
                      blocks=[np.zeros(24 * 8192, np.complex64)])
    assert rc == 0
    lines = [ln for ln in out.getvalue().splitlines() if ln.startswith("BIS ")]
    assert len(lines) == int((bis["status"] == bo.OK).sum()) and all(len(ln.split()) == 9 for ln in lines)
    bigs = messages.ble_broadcast_iso(bis)
    assert lines[0] == formats.bis_line(bigs[0], bigs[0]["streams"][0], bigs[0]["streams"][0]["pdus"][0]).strip()
    data = pcap.read_bytes()
    assert data.startswith(formats.PCAP_HDR_BLE) and data.endswith(formats.ble_pcap_bis_block(bis))
