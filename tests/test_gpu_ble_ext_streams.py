"""snrx_ble_aux and snrx_ble_coded driven with constructed bit streams (snrx_debug_process_bits) and held to
oracle/aux_oracle.py and oracle/coded_oracle.py at every edge of their contracts.

Every decision of a wideband batch passes through the channelizer, so no IQ construction can force the slicer bits at a window
edge, a tie or a truncation residue.  The test hook puts chosen words where the channelizer would have left them.  One list of
cases carries the constructions of tests/test_ble_aux.py and tests/test_ble_coded.py, replayed with depth-0 sources taken from
the engine's own poll, and the edges that exist only in the kernels: the scan's 2048-position tiles and their halo, the
window kernel's lane stride, the decode kernel's 8-lane groups sharing a warp, the search's 32-word passes and the ballot
steps of `first`.

The unmarked test runs every case through the oracles and asserts that its edge fires (status, sample_index, tie winner);
the gpu tests feed the same words to the engine and require its lists to equal the oracles' field for field."""
from __future__ import annotations

import functools
from ctypes import byref, c_uint32, c_void_p
from typing import Callable, NamedTuple

import numpy as np
import pytest

import ble_bits as bb
from conftest import assert_frames_equal
from oracle import aux_oracle as ao
from oracle import coded_oracle as co
from snout_b200 import _abi, synth
from test_ble_aux import Batch, _chain, aux_pdu, aux_symbols, plant_stride, primary_record
from test_ble_coded import coded_decisions, coded_primary_with_ptr, packet_end, plant, prim_pdu, tie_stream
from test_gpu_ble_aux import assert_aux_equal
from test_gpu_ble_coded import assert_coded_equal

TILE = 2048                                   # k_ble_coded_scan positions per block
N_CH = 40


# ------------------------------------------------------------------------------------------------ cases
class Case(NamedTuple):
    name: str
    kind: str                                 # "aux" | "coded"
    words: np.ndarray                         # uint32 [captures, 40, words]
    n_out: int                                # channel samples per capture (n_samples = 24 n_out)
    check: Callable                           # the expectation on the oracle's list (the edge fires)
    shard: tuple | None = None                # (pre_out, first_window, n_windows or 0) in channel samples
    first_capture: int = 0
    frames: np.ndarray | None = None          # aux: the synthetic ADV_EXT_IND records the CPU construction meant
    spots: tuple = ()                         # aux: (capture, channel, s) of the planted ADV_EXT_INDs

    def geo(self) -> dict:
        pre, w0, nw = self.shard or (0, 0, 0)
        return dict(first_window=w0, pre_out=pre, first_capture=self.first_capture)

    def shard_arg(self) -> dict:
        pre, w0, nw = self.shard or (0, 0, 0)
        return dict(pre_samples=24 * pre, body_samples=24 * 8192 * nw, first_window=w0, first_capture_id=self.first_capture)

    def coded_list(self):
        pre, w0, nw = self.shard or (0, 0, 0)
        return co.coded_list(self.words, self.n_out, n_windows=nw or None, **self.geo())

    def aux_list(self, frames):
        return ao.aux_list(self.words, frames, self.n_out, **self.geo())


def words_of(batches) -> np.ndarray:
    """[captures, 40, words] of Batch objects of one length; the last decision of every stream is 0, as the front end
    leaves it (ble_bits.effective_bits), so that the legacy oracle on bits_to_iq sees the same streams."""
    w = np.concatenate([b.words() for b in batches])
    n = batches[0].n
    w[:, :, 4 + (n - 1) // 32] &= ~np.uint32(1 << ((n - 1) % 32))
    return w


def coded_case(name, bts, check, **kw) -> Case:
    bts = bts if isinstance(bts, list) else [bts]
    return Case(name, "coded", words_of(bts), bts[0].n, check, **kw)


def aux_case(name, bt: Batch, check, shard=None) -> Case:
    """bt.frames: primary_record()s of the CPU construction.  Each is planted as a real ADV_EXT_IND at its sample_index on
    its channel, so that the engine's own poll provides it."""
    spots = []
    for f in bt.frames:
        s, ch = int(f["sample_index"]), int(f["channel"])
        pdu = bytes(f["bytes"][: int(f["len"]) - 3])
        plant_stride(bt.b[ch], s, bb.frame_symbols(ch, pdu[:2], pdu[2:]), 4)
        spots.append((0, ch, s))
    fr = np.array(bt.frames, dtype=_abi.FRAME_DTYPE)
    return Case(name, "aux", words_of([bt]), bt.n, check, shard=shard, frames=fr, spots=tuple(spots))


def zeroed(n, seed=0, chans=(37, 38, 39)) -> Batch:
    bt = Batch(n, seed=seed)
    for c in chans:
        bt.b[c] &= 0
    return bt


def planted(got, spots):
    keep = (got["depth"] > 0) | np.isin(got["sample_index"], list(spots))
    return got[keep], np.nonzero(keep)[0]


def ok_decoded(r, channel, pdu, crc_ok=True):
    want = pdu + synth.ble_crc24(pdu)
    assert r["status"] == ao.OK and r["channel"] == channel and bool(r["crc_ok"]) == crc_ok
    assert r["len"] == len(want) and (not crc_ok or bytes(r["bytes"][: len(want)]) == want)


# ------------------------------------------------------------------------------------------------ B: aux
def _aux_window_edges():
    out = []
    for ca in (0, 1):
        for units, offset in ((30, 0), (30, 8191), (300, 0), (300, 8191), (30, 517)):
            rng = np.random.default_rng(units + offset + ca)
            lo, hi = ao.window(units, offset, ca)
            s = 300
            for where, found in ((lo, True), (hi, True), (lo - 1, False), (hi + 1, False)):
                bt = Batch(s + hi + 2000, seed=offset + where)
                pdu = aux_pdu(rng, 20)
                bt.b[9] &= 0
                plant_stride(bt.b[9], s + where, aux_symbols(9, pdu), 4)
                bt.frames.append(primary_record(s, synth.aux_ptr_bytes(9, ca, units, offset, 0)))

                def check(got, s=s, lo=lo, hi=hi, where=where, found=found, pdu=pdu):
                    (r,) = got
                    assert (r["win_lo"], r["win_hi"]) == (s + lo, s + hi)
                    if found:
                        ok_decoded(r, 9, pdu)
                        assert r["sample_index"] == s + where
                    else:
                        assert r["status"] == ao.NOT_FOUND
                out.append(aux_case(f"aux window ca{ca} {units}/{offset} at {where}", bt, check))
    return out


def _aux_2m_phases():
    out = []
    for phase in (0, 1):
        rng = np.random.default_rng(phase)
        bt = Batch(6000, seed=phase)
        s = 500
        lo, hi = ao.window(30, 20, 1)
        a, b_ = s + lo + 10 + phase, s + lo + 41 + phase
        p1, p2 = aux_pdu(rng, 30), aux_pdu(rng, 40)
        plant_stride(bt.b[3], b_, aux_symbols(3, p2), 2)
        plant_stride(bt.b[3], a, aux_symbols(3, p1), 2)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(3, 1, 30, 20, 1)))

        def check(got, a=a, p1=p1):
            (r,) = got
            ok_decoded(r, 3, p1)
            assert r["sample_index"] == a and r["phy"] == ao.PHY_2M
        out.append(aux_case(f"aux 2M phase {phase}, earliest match", bt, check))
    return out


def _aux_every_length():
    rng = np.random.default_rng(7)
    bt = Batch(2_300_000, seed=7)
    s, want = 100, []
    for ln in range(256):
        sps = 4 if ln % 2 == 0 else 2
        pdu = synth.ext_pdu(b"", bytes(rng.integers(0, 256, ln, dtype=np.uint8))) if ln < 2 else aux_pdu(rng, max(ln, 12))[:2 + ln]
        pdu = bytes([pdu[0], ln]) + pdu[2:2 + ln]
        ok = ln % 5 != 3
        lo, _ = ao.window(30, 3, 0)
        plant_stride(bt.b[11], s + lo + 8, aux_symbols(11, pdu, ok), sps)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(11, 0, 30, 3, sps == 2)))
        want.append((pdu, ok))
        s += lo + 8 + sps * (40 + 8 * (ln + 5)) + 600            # room for the planted ADV_EXT_IND (512 samples)

    def check(got):
        assert len(got) == 256
        for r, (pdu, ok) in zip(got, want):
            ok_decoded(r, 11, pdu, ok)
    return [aux_case("aux every length, CRC errors", bt, check)]


def _aux_buffer_end():
    out = []
    rng = np.random.default_rng(3)
    pdu = aux_pdu(rng, 100)
    nbits = 32 + 8 * (len(pdu) + 3)
    for sps in (4, 2):
        lo, hi = ao.window(30, 10, 1)                           # (offset 2 in the CPU test: the ADV_EXT_IND must fit too)
        s = 1000
        at = s + hi - 10
        end = at + (nbits - 1) * sps
        ptr = synth.aux_ptr_bytes(30, 1, 30, 10, sps == 2)
        ns = [(end + 2, ao.OK), (end + 1, ao.TRUNCATED)]
        ns += [(at + 47 * sps + 2 + r, ao.TRUNCATED) for r in range(-1, 3)]   # the header's last decision, both sides
        for n, status in ns:
            bt = Batch(n, seed=n)
            plant_stride(bt.b[30], at, aux_symbols(30, pdu), sps)
            bt.frames.append(primary_record(s, ptr))

            def check(got, status=status, at=at, n=n, sps=sps):
                (r,) = got
                assert r["status"] == status
                if status == ao.TRUNCATED:
                    assert r["sample_index"] == at and r["len"] == 0
            out.append(aux_case(f"aux end sps{sps} n_out {n}", bt, check))
        for extra, outside in ((1, True), (2, False)):
            bt = Batch(s + hi + 31 * sps + extra, seed=1)
            bt.frames.append(primary_record(s, ptr))
            out.append(aux_case(f"aux OUTSIDE sps{sps} +{extra}", bt,
                                lambda got, outside=outside: (got[0]["status"] == ao.OUTSIDE) == outside or pytest.fail("edge")))
    return out


def _aux_unsearched():
    bt = Batch(6000)
    for j, ptr in enumerate((synth.aux_ptr_bytes(5, 0, 30, 3, 2), synth.aux_ptr_bytes(5, 0, 30, 3, 3),
                             synth.aux_ptr_bytes(37, 0, 30, 3, 0))):
        bt.frames.append(primary_record(100 + 600 * j, ptr, channel=37 + j))

    def check(got):
        assert list(got["status"]) == [ao.UNSUPPORTED_PHY, ao.UNSUPPORTED_PHY, ao.BAD_CHANNEL]
    return [aux_case("aux statuses not searched", bt, check)]


def _aux_chains():
    out = []
    for links in (1, 2, 5, 15, 16, 17):
        rng = np.random.default_rng(links)
        bt = Batch(2000 + 3000 * (links + 2), seed=links)
        chans = [int(c) for c in rng.integers(0, 37, links)]
        phys = [int(p) for p in rng.integers(0, 2, links)]
        starts, pdus, ptr0 = _chain(bt, rng, 100, chans, phys)
        bt.frames.append(primary_record(100, ptr0))

        def check(got, links=links, chans=chans, pdus=pdus, starts=starts):
            n_ok = min(links, ao.MAX_DEPTH + 1)
            assert len(got) == n_ok + (1 if links > ao.MAX_DEPTH + 1 else 0)
            for d in range(n_ok):
                ok_decoded(got[d], chans[d], pdus[d])
                assert got[d]["depth"] == d and got[d]["sample_index"] == starts[d]
            if links > ao.MAX_DEPTH + 1:
                assert got[-1]["status"] == ao.DEPTH_LIMIT and got[-1]["depth"] == ao.MAX_DEPTH + 1
        out.append(aux_case(f"aux chain of {links}", bt, check))
    rng = np.random.default_rng(5)
    bt = Batch(20000, seed=5)
    starts, pdus, ptr0 = _chain(bt, rng, 100, [4, 9], [0, 1], loop_last=True)
    bt.frames.append(primary_record(100, ptr0))

    def check_loop(got):
        assert len(got) == 3 and got[2]["sample_index"] == got[1]["sample_index"] and got[2]["first"] == 1
    out.append(aux_case("aux chain pointing back at itself", bt, check_loop))
    rng = np.random.default_rng(9)
    bt = Batch(40000, seed=9)
    starts, pdus, _ = _chain(bt, rng, 9000, [17, 2], [1, 0])
    for j, s in enumerate((1000, 4000, 7000)):
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(17, 0, 30, (starts[0] - s) // 4 // 30, 1), channel=37 + j))

    def check_three(got):
        assert list(got["depth"]) == [0, 0, 0, 1] and list(got["first"]) == [0, 0, 0, 3]
        ok_decoded(got[3], 2, pdus[1])
    out.append(aux_case("aux three primaries, one packet", bt, check_three))
    return out


def _aux_shards():
    """test_ble_aux's shard construction, with a pre halo of one window (128 in the CPU test: any multiple of 128 is
    valid) so that the ADV_EXT_IND record lies in the shard's body."""
    out = []
    rng = np.random.default_rng(11)
    whole = Batch(60000, seed=11)
    pdu = aux_pdu(rng, 60)
    s = 20000
    at = s + ao.window(30, 30, 1)[0] + 20
    plant_stride(whole.b[6], at, aux_symbols(6, pdu), 4)
    whole.frames.append(primary_record(s, synth.aux_ptr_bytes(6, 1, 30, 30, 0)))
    ref = aux_case("aux whole", whole, lambda got: ok_decoded(got[0], 6, pdu))
    out.append(ref)
    pre, w0 = 128, 2
    hi = s + ao.window(30, 30, 1)[1]
    for end, status in ((60000, ao.OK), (at + 900, ao.TRUNCATED), (hi + 100, ao.OUTSIDE)):
        a = 8192 * w0 - pre
        sh = Batch(end - a)
        for c in list(whole.b):
            sh.b[c] = whole.b[c][a:end].copy()
        w = words_of([sh])
        fr = ref.frames

        def check(got, status=status):
            assert got[0]["status"] == status
        out.append(Case(f"aux shard to {end}", "aux", w, sh.n, check, shard=(pre, w0, 0), frames=fr, spots=ref.spots))
    return out


# ------------------------------------------------------------------------------------------------ D: aux kernel edges
def _aux_kernel_edges():
    out = []
    rng = np.random.default_rng(60)
    s = 600
    lo, hi = ao.window(300, 0, 1)                             # 300 us units: a window of ~1220 samples, ~38 words
    assert hi - lo > 32 * 33
    for name, at_rel, sps in (("second pass", 32 * ((s + lo) // 32 + 34) + 3 - s, 4),
                              ("bit 0", 32 * ((s + lo) // 32 + 5) - s, 4),
                              ("bit 31", 32 * ((s + lo) // 32 + 5) + 31 - s, 4),
                              ("2M across words", 32 * ((s + lo) // 32 + 7) + 20 - s, 2)):
        assert lo <= at_rel <= hi
        bt = Batch(s + hi + 4000, seed=at_rel)
        bt.b[13] &= 0
        pdu = aux_pdu(rng, 24)
        plant_stride(bt.b[13], s + at_rel, aux_symbols(13, pdu), sps)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(13, 1, 300, 0, sps == 2)))

        def check(got, at=s + at_rel, pdu=pdu):
            (r,) = got
            ok_decoded(r, 13, pdu)
            assert r["sample_index"] == at
        out.append(aux_case(f"aux search {name}", bt, check))
    # k_ble_aux_first: 34 pointers find nothing, then three find one packet: `first` is found in the ballot's second step
    rng = np.random.default_rng(61)
    n_lead, n_hit = 34, 3
    target = 600 * (n_lead + n_hit) + 4000
    bt = Batch(target + 10000, seed=61)
    bt.b[5] &= 0
    bt.b[17] &= 0
    chain = aux_pdu(rng, 20)
    chain_at = target + 3000
    head = aux_pdu(rng, 30, synth.aux_ptr_bytes(22, 1, 30, (chain_at - target) // 120, 0))
    plant_stride(bt.b[17], target, aux_symbols(17, head), 4)
    plant_stride(bt.b[22], chain_at, aux_symbols(22, chain), 4)
    for j in range(n_lead + n_hit):
        s = 200 + 600 * j
        ch = 5 if j < n_lead else 17
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(ch, 1, 30, (target - s) // 120, 0)))

    def check_first(got):
        assert len(got) == n_lead + n_hit + 1
        assert (got["status"][:n_lead] == ao.NOT_FOUND).all()
        assert list(got["first"][n_lead:n_lead + n_hit]) == [n_lead] * n_hit
        assert got[-1]["depth"] == 1 and got[-1]["parent"] == n_lead
        ok_decoded(got[-1], 22, chain)
    out.append(aux_case("aux first past 32 entries", bt, check_first))
    return out


# ------------------------------------------------------------------------------------------------ C: Long Range
def _coded_round_trips():
    out = []
    for s in (8, 2):
        rng = np.random.default_rng(s)
        step = 4 if s == 8 else 1
        for lo in range(0, 256, 64):
            lengths = list(range(lo, lo + 64, step)) + ([255] if lo == 192 and step > 1 else [])
            ends = [0]
            for ln in lengths:
                ends.append(packet_end(ends[-1] + 300, ln, s) + 40)
            bt = Batch(ends[-1] + 2000, seed=lo + s)
            want = []
            for ln, n0 in zip(lengths, ends[:-1]):
                pdu = bytes([int(rng.integers(0, 256)) & 0xEF, ln]) + bytes(rng.integers(0, 256, ln, dtype=np.uint8))
                plant(bt.b[37], n0 + 300, coded_decisions(pdu, 37, s))
                want.append((n0 + 300, pdu))

            def check(got, want=want, s=s):
                ok = got[(got["status"] == co.OK) & (got["crc_ok"] == 1)]
                assert [int(r["sample_index"]) for r in ok] == [n for n, _ in want]
                for r, (n, pdu) in zip(ok, want):
                    ok_decoded(r, 37, pdu)
                    assert r["ci"] == (0 if s == 8 else 1) and r["metric"] == 0
            out.append(coded_case(f"coded round trip S={s} lengths {lo}..", bt, check))
    return out


def _coded_threshold_and_ties():
    out = []
    for extra in (0, 1):
        rng = np.random.default_rng(3)
        bt = zeroed(8000, 3)
        n = 3000
        clean = coded_decisions(prim_pdu(rng), 37, 8)
        for seed in range(200):
            dec = clean.copy()
            dec[np.random.default_rng(seed).choice(co.AA_SAMPLES, 400 + extra, replace=False)] ^= 1
            plant(bt.b[37], n, dec)
            d = co.distances(bt.b[37], bt.n)
            if (np.r_[d[n - 16:n], d[n + 1:n + 17]] > 401).all():
                break
        assert d[n] == 400 + extra
        out.append(coded_case(f"coded d = T + {extra}", bt,
                              lambda got, extra=extra: ((3000 in got["sample_index"]) == (extra == 0)) or pytest.fail("edge")))
    for seed in range(4):
        n, k, b = tie_stream(seed)
        bt = Batch(len(b), seed=seed)
        bt.b[38] = b

        def check(got, n=n, k=k):
            hits = list(got["sample_index"][got["channel"] == 38])
            assert n in hits and n + k not in hits
        out.append(coded_case(f"coded minimum tie seed {seed} (k = {k})", bt, check))
    bt = Batch(400_000, seed=77)
    for c in (37, 38, 39):
        bt.b[c]
    out.append(coded_case("coded random streams", bt, lambda got: len(got) == 0 or pytest.fail("packets")))
    return out


def _coded_viterbi_and_ci():
    out = []
    for s in (8, 2):
        rng = np.random.default_rng(11 + s)
        L = 16 if s == 8 else 4
        pdu = prim_pdu(rng, extra=10)
        dec = coded_decisions(pdu, 37, s).copy()
        for k in list(range(40, 56)) + list(range(150, 152)) + [230]:
            seg = dec[co.BLOCK2 + k * L:co.BLOCK2 + (k + 1) * L]
            seg[:] = np.r_[np.ones(L // 2), np.zeros(L // 2)].astype(np.uint8) if s == 2 else np.tile([0, 1], L // 2).astype(np.uint8)
        bt = zeroed(40000, 5)
        plant(bt.b[37], 1000, dec)

        def check(got, pdu=pdu):
            (r,) = got[got["sample_index"] == 1000]
            assert r["status"] == co.OK and bytes(r["bytes"][: r["len"]]) != pdu + synth.ble_crc24(pdu)
        out.append(coded_case(f"coded Viterbi ties S={s}", bt, check))
    rng = np.random.default_rng(4)
    pdu = prim_pdu(rng)
    bt = zeroed(60000, 4)
    for v in range(4):
        plant(bt.b[37], 1000 + 12000 * v, coded_decisions(pdu, 37, 8, ci=v))

    def check_ci(got):
        g, _ = planted(got, [1000 + 12000 * v for v in range(4)])
        assert list(g["ci"]) == [0, 1, 2, 3] and list(g["status"]) == [co.OK, co.OK, co.RESERVED_CI, co.RESERVED_CI]
    out.append(coded_case("coded CI values", bt, check_ci))
    for a, b_ in ((0, 1), (1, 3), (2, 3), (0, 2)):
        dec = coded_decisions(pdu, 37, 8, ci=a).copy()
        pa, pb = co.CI_PATTERNS[a], co.CI_PATTERNS[b_]
        diff = np.nonzero(pa != pb)[0]
        dec[co.AA_SAMPLES + diff[: len(diff) // 2]] = pb[diff[: len(diff) // 2]]
        bt = zeroed(30000, a)
        plant(bt.b[37], 1000, dec)
        out.append(coded_case(f"coded CI tie {a}/{b_}", bt,
                              lambda got, m=min(a, b_): int(planted(got, [1000])[0][0]["ci"]) == m or pytest.fail("tie")))
    return out


def _coded_truncation():
    out = []
    for s in (8, 2):
        rng = np.random.default_rng(s + 20)
        pdu = prim_pdu(rng, extra=5)
        ln, L, ci = pdu[1], (16 if s == 8 else 4), (0 if s == 8 else 1)
        n = 600
        edges = (("ci", n + co.BLOCK2 - 1), ("hdr", n + co.BLOCK2 + 80 * L - 1), ("full", packet_end(n, ln, s)))
        for edge, last in edges:
            for r in range(16):
                n_out = last + 2 - 8 + r
                bt = zeroed(n_out, r)
                plant(bt.b[37], n, coded_decisions(pdu, 37, s))

                def check(got, edge=edge, usable=n_out - 2 >= last, ci=ci, ln=ln):
                    g, _ = planted(got, [600])
                    (g,) = g
                    if edge == "ci":
                        assert g["status"] == co.TRUNCATED and g["ci"] == (ci if usable else 0xFF)
                    elif edge == "hdr":
                        assert g["status"] == co.TRUNCATED and g["ci"] == ci and g["len"] == 0
                    else:
                        assert g["status"] == (co.OK if usable else co.TRUNCATED) and g["len"] == (ln + 5 if usable else 0)
                out.append(coded_case(f"coded truncation S={s} {edge} r{r}", bt, check))
    return out


def _coded_last_position_and_windows():
    out = []
    rng = np.random.default_rng(30)
    pdu = prim_pdu(rng)
    n = 5000
    for n_out, found in ((n + co.AA_SAMPLES + 1, True), (n + co.AA_SAMPLES, False)):
        bt = zeroed(n_out, 1)
        plant(bt.b[37], n, coded_decisions(pdu, 37, 8))
        out.append(coded_case(f"coded last defined position {found}", bt,
                              lambda got, found=found, n=n: ((n in got["sample_index"]) == found) or pytest.fail("edge")))
    units, off, ca = 30, 40, 1
    lo, hi = ao.window(units, off, ca)
    src = 1000
    win_hi = src + hi
    for extra, status in ((0, co.TRUNCATED), (-1, co.OUTSIDE)):
        bt = zeroed(win_hi + co.AA_SAMPLES + 1 + extra, 2, (37, 38, 39, 9))
        coded_primary_with_ptr(rng, bt, src, synth.aux_ptr_bytes(9, ca, units, off, 2))
        plant(bt.b[9], win_hi, coded_decisions(aux_pdu(rng, 20), 9, 8))

        def check(got, status=status):
            g, _ = planted(got, [src])
            assert len(g) == 2 and g[1]["win_hi"] == win_hi and g[1]["status"] == status
        out.append(coded_case(f"coded target at the last defined position, {extra}", bt, check))
    for dst_phy in (0, 1, 2):
        for where in ("lo", "hi", "lo-1", "hi+1"):
            rng = np.random.default_rng(100 * dst_phy + len(where) + (where[-1] == "1"))
            n = 2000
            shift = -320 + co.PREAMBLE[dst_phy]
            at = n + shift + {"lo": lo, "hi": hi, "lo-1": lo - 1, "hi+1": hi + 1}[where]
            bt = zeroed(n + hi + 40000, dst_phy, (37, 38, 39, 9))
            coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(9, ca, units, off, dst_phy))
            target = aux_pdu(rng, 30)
            if dst_phy == 2:
                plant(bt.b[9], at, coded_decisions(target, 9, 2))
            else:
                plant_stride(bt.b[9], at, aux_symbols(9, target), 2 if dst_phy == 1 else 4)

            def check(got, where=where, at=at, target=target, dst_phy=dst_phy, n=n):
                g, _ = planted(got, [n])
                assert len(g) == 2
                if where in ("lo", "hi"):
                    ok_decoded(g[1], 9, target)
                    assert g[1]["sample_index"] == at
                elif dst_phy == 2:
                    assert g[1]["sample_index"] == (g[1]["win_lo"] if where == "lo-1" else g[1]["win_hi"])
                else:
                    assert g[1]["status"] == co.NOT_FOUND
            out.append(coded_case(f"coded window PHY {dst_phy} at {where}", bt, check))
    return out


def _coded_pointers():
    out = []
    for src_phy in (0, 1):
        rng = np.random.default_rng(src_phy + 40)
        bt = zeroed(80000, src_phy, (37, 38, 39, 4, 21))
        n = 1000
        lo1, _ = ao.window(30, 100, 1)
        a1 = n - 320 + 32 + lo1 + 50
        _, hi2 = ao.window(30, 60, 1)
        a2 = a1 - 32 + 320 + hi2
        link = aux_pdu(rng, 20, synth.aux_ptr_bytes(21, 1, 30, 60, 2))
        plant_stride(bt.b[4], a1, aux_symbols(4, link), 2 if src_phy else 4)
        coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(4, 1, 30, 100, src_phy))
        last = aux_pdu(rng, 12)
        plant(bt.b[21], a2, coded_decisions(last, 21, 8))

        def check(got, a2=a2, last=last, n=n):
            g, _ = planted(got, [n])
            assert len(g) == 3 and g[2]["sample_index"] == a2 and g[2]["depth"] == 2
            ok_decoded(g[2], 21, last)
        out.append(coded_case(f"coded uncoded source PHY {src_phy} to Coded", bt, check))
    rng = np.random.default_rng(8)
    bt = zeroed(120000, 8, (37, 38, 39, 17))
    target_at = 60000
    target = aux_pdu(rng, 25)
    plant(bt.b[17], target_at, coded_decisions(target, 17, 2))
    for j, n in enumerate((2000, 20000, 38000)):
        coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(17, 1, 30, (target_at - n) // 120, 2), channel=37 + j)
    bt.b[37][100_000:] = 0
    coded_primary_with_ptr(rng, bt, 100_000, synth.aux_ptr_bytes(17, 1, 300, 8000, 2))

    def check_three(got):
        g, idx = planted(got, [2000, 20000, 38000, 100_000])
        assert list(g["depth"]) == [0, 0, 0, 0, 1, 1, 1, 1] and g[5]["status"] == co.OUTSIDE
        assert list(g["first"][4:]) == [idx[4], idx[5], idx[4], idx[4]]
    out.append(coded_case("coded three primaries, one packet", bt, check_three))
    # the depth limit: 16 pointed packets are followed, the 17th pointer is DEPTH_LIMIT
    rng = np.random.default_rng(12)
    links = 17
    bt = zeroed(2000 + 3000 * (links + 3), 12)
    starts = [4000 + 3000 * k for k in range(links)]
    coded_primary_with_ptr(rng, bt, 500, synth.aux_ptr_bytes(3, 1, 30, (starts[0] - (500 - 320 + 32)) // 120, 0))
    for k in range(links):
        ptr = synth.aux_ptr_bytes(3 + (k + 1) % 30, 1, 30, (starts[k + 1] - starts[k]) // 120, 0) if k + 1 < links else None
        plant_stride(bt.b[3 + k % 30], starts[k], aux_symbols(3 + k % 30, aux_pdu(rng, 20, ptr)), 4)

    def check_depth(got):
        g, _ = planted(got, [500])
        assert len(g) == 1 + co.MAX_DEPTH + 1 and g[-1]["status"] == co.DEPTH_LIMIT
        assert all(g[d]["status"] == co.OK and g[d]["crc_ok"] for d in range(1, co.MAX_DEPTH + 1))
    out.append(coded_case("coded depth limit 16 / 17", bt, check_depth))
    # `first` compares the PHY: a Coded target and a 1M target found at the same sample of one channel are two packets
    rng = np.random.default_rng(14)
    bt = zeroed(60000, 14, (37, 38, 39, 9))
    tgt = 30000
    dec = coded_decisions(aux_pdu(rng, 20), 9, 8).copy()
    plant(bt.b[9], tgt, dec)
    plant_stride(bt.b[9], tgt, bb.aa_bits(ao.ADV_AA), 4)       # the 1M access address over the coded one: d(tgt) <= 32
    for j, (n, phy) in enumerate(((2000, 2), (8000, 0), (14000, 2))):
        coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(9, 1, 30, (tgt - n + 320 - co.PREAMBLE[phy]) // 120, phy),
                               channel=37 + j)

    def check_phy(got):
        g, idx = planted(got, [2000, 8000, 14000])
        t = g[g["depth"] == 1]
        assert list(t["sample_index"]) == [tgt] * 3 and list(t["phy"]) == [2, 0, 2]
        k = idx[g["depth"] == 1]
        assert list(t["first"]) == [k[0], k[1], k[0]]
    out.append(coded_case("coded first compares the PHY", bt, check_phy))
    return out


def _coded_shards():
    out = []
    rng = np.random.default_rng(13)
    whole = zeroed(8192 * 12, 13)
    spots = [100, 8192 * 3 - 30, 8192 * 3 + 5, 8192 * 6 - 1100, 8192 * 9 + 17]
    for k, n in enumerate(spots):
        plant(whole.b[37 + k % 3], n, coded_decisions(prim_pdu(rng), 37 + k % 3, 8 if k % 2 else 2))
    ref = co.coded_list(words_of([whole]), whole.n)
    want = planted(ref, spots)[0]
    key = ("sample_index", "channel", "status", "ci", "len", "crc_ok", "aa_errors", "metric", "bytes")
    for w0, w1 in ((0, 3), (3, 6), (6, 9), (9, 12)):
        pre = 128 if w0 else 0
        a, b = 8192 * w0 - pre, min(whole.n, 8192 * w1 + 9000)
        sh = Batch(b - a)
        for c in list(whole.b):
            sh.b[c] = whole.b[c][a:b].copy()

        def check(got, w0=w0, w1=w1):
            assert all(8192 * w0 <= int(r["sample_index"]) < 8192 * w1 for r in got)
            mine = {tuple(np.asarray(r[k]).tobytes() for k in key) for r in planted(got, spots)[0]}
            inside = {tuple(np.asarray(r[k]).tobytes() for k in key) for r in want if 8192 * w0 <= r["sample_index"] < 8192 * w1}
            assert mine == inside
        out.append(coded_case(f"coded shard {w0}..{w1}", sh, check, shard=(pre, w0, w1 - w0), first_capture=3 * w0))
    return out


# ------------------------------------------------------------------------------------------------ D: Long Range kernel edges
def _clean(n_out, chans=(37, 38, 39)):
    return zeroed(n_out, n_out % 1000, chans)


def _coded_kernel_edges():
    out = []
    rng = np.random.default_rng(70)
    pdu = prim_pdu(rng)
    for k in (1, 3):                                            # k_ble_coded_scan: tile edges
        for o in (-1, 0, 1):
            n = TILE * k + o
            bt = _clean(n + 12000)
            plant(bt.b[38], n, coded_decisions(pdu, 38, 2))
            out.append(coded_case(f"coded scan at {TILE}*{k}{o:+d}", bt,
                                  lambda got, n=n: list(got["sample_index"]) == [n] or pytest.fail(str(got["sample_index"]))))
    for seed in range(2):                                       # tie pairs straddling a tile boundary, on either side
        n, k, b = tie_stream(seed)
        for o in (-k, -1, 0, -16, 16 - k):
            at = 3 * TILE + o
            bt = Batch(at + 3000, seed=seed)
            bt.b[39] = np.r_[np.random.default_rng(seed).integers(0, 2, at - n).astype(np.uint8), b][: bt.n]

            def check(got, at=at, k=k):
                hits = list(got["sample_index"][got["channel"] == 39])
                assert at in hits and at + k not in hits
            out.append(coded_case(f"coded tie across a tile, seed {seed} k {k} at {o:+d}", bt, check))
    n_out = 5 * TILE + 1300                                     # the last tile is partial
    bt = _clean(n_out)
    plant(bt.b[37], 5 * TILE + 200, coded_decisions(pdu, 37, 8))
    plant(bt.b[39], 2 * TILE + 7, coded_decisions(pdu, 39, 2))
    out.append(coded_case("coded primary in the last partial tile", bt,
                          lambda got: 5 * TILE + 200 in got["sample_index"] or pytest.fail("missing")))
    # three captures: stream -> (capture, channel), first_capture_id 7
    bts = []
    for cap in range(3):
        bt = _clean(30000)
        for j, ch in enumerate((37, 38, 39)):
            if (cap + j) % 2 == 0:
                plant(bt.b[ch], 1000 + 3000 * cap + 500 * j, coded_decisions(pdu, ch, 2))
        bts.append(bt)

    def check_caps(got):
        ok = got[(got["status"] == co.OK) & (got["crc_ok"] == 1)]
        want = [(7 + cap, ch, 1000 + 3000 * cap + 500 * j) for cap in range(3) for j, ch in enumerate((37, 38, 39)) if (cap + j) % 2 == 0]
        assert [(int(r["capture_id"]), int(r["channel"]), int(r["sample_index"])) for r in ok] == want
    out.append(coded_case("coded three captures", bts, check_caps, first_capture=7))
    # a shard's body: primaries at body_lo, body_hi - 1 (reported) and body_hi (not)
    pre, w0 = 128, 1
    bt = _clean(pre + 8192 + 12000)
    for ch, n in ((37, pre), (38, pre + 8191), (39, pre + 8192)):
        plant(bt.b[ch], n, coded_decisions(pdu, ch, 2))
    out.append(coded_case("coded shard body edges", bt,
                          lambda got: ({8192, 16383} <= set(got["sample_index"].tolist()) and got["sample_index"].max() < 16384)
                          or pytest.fail("body"),
                          shard=(pre, w0, 1)))
    # k_ble_coded_window: 32 lanes stride over the window; equal d -> the earlier n, a cleaner later copy -> the later
    lo, hi = ao.window(300, 1, 1)
    src = 1000
    for gap in (1056, 1029, None):                             # same lane, different lanes, one copy past the first 32
        for later_cleaner in ((False, True) if gap else (False,)):
            bt = _clean(src + hi + 6000, (37, 38, 39, 9))
            coded_primary_with_ptr(rng, bt, src, synth.aux_ptr_bytes(9, 1, 300, 1, 2))
            n1 = src + lo + 40
            tgt = aux_pdu(rng, 20)
            copy = co.PATTERN.copy()
            if gap:
                first = copy.copy()
                if later_cleaner:
                    first[[5, 300, 700]] ^= 1
                plant(bt.b[9], n1, first)
                plant(bt.b[9], n1 + gap, coded_decisions(tgt, 9, 2))
                want = n1 + gap if later_cleaner else n1
            else:
                plant(bt.b[9], n1, coded_decisions(tgt, 9, 2))
                want = n1

            def check(got, want=want):
                g, _ = planted(got, [src])
                assert len(g) == 2 and g[1]["sample_index"] == want
            out.append(coded_case(f"coded window gap {gap} later cleaner {later_cleaner}", bt, check))
    # k_ble_coded_decode: consecutive primaries of every outcome, groups of one warp on different paths
    bts, n_out = [], 16000
    L8, L2 = 16, 4
    p_short = prim_pdu(rng)
    p_long = prim_pdu(rng, extra=30)
    for cap in range(2):
        bt = _clean(n_out)
        plant(bt.b[37], 300, coded_decisions(p_short, 37, 2))                         # S=2 OK
        plant(bt.b[37], 3000, coded_decisions(p_short, 37, 8, ci=2))                  # reserved CI (S=8 AA and CI)
        plant(bt.b[37], 5000, coded_decisions(p_short, 37, 2))                        # S=2 OK
        plant(bt.b[37], n_out - 2 - co.BLOCK2 - 80 * L2 - 200, coded_decisions(p_long, 37, 2))   # in the full run
        plant(bt.b[38], n_out - 2 - co.BLOCK2 - 40 * L8, coded_decisions(p_long, 38, 8))         # in the header run
        plant(bt.b[39], 900, coded_decisions(p_short, 39, 2))
        plant(bt.b[39], n_out - 2 - co.AA_SAMPLES - 60, coded_decisions(p_long, 39, 2))          # before CI
        bts.append(bt)

    def check_mix(got):
        want = {(37, 300): (co.OK, 1), (37, 3000): (co.RESERVED_CI, 2), (37, 5000): (co.OK, 1), (39, 900): (co.OK, 1),
                (37, n_out - 2 - co.BLOCK2 - 80 * L2 - 200): (co.TRUNCATED, 1),
                (38, n_out - 2 - co.BLOCK2 - 40 * L8): (co.TRUNCATED, 0),
                (39, n_out - 2 - co.AA_SAMPLES - 60): (co.TRUNCATED, 0xFF)}
        for cap in range(2):
            g = {(int(r["channel"]), int(r["sample_index"])): (int(r["status"]), int(r["ci"])) for r in got if r["capture_id"] == cap}
            assert all(g[k] == v for k, v in want.items()), g
        assert len(got) >= 32                                    # (with the false primaries of the S=8 bodies)
    out.append(coded_case("coded decode outcomes mixed in one warp", bts, check_mix))
    return out


def all_cases() -> list[Case]:
    cases = []
    for f in (_aux_window_edges, _aux_2m_phases, _aux_every_length, _aux_buffer_end, _aux_unsearched, _aux_chains,
              _aux_shards, _aux_kernel_edges, _coded_round_trips, _coded_threshold_and_ties, _coded_viterbi_and_ci,
              _coded_truncation, _coded_last_position_and_windows, _coded_pointers, _coded_shards, _coded_kernel_edges):
        cases += f()
    assert len({c.name for c in cases}) == len(cases)
    return cases


@functools.lru_cache(maxsize=None)
def cases() -> list[Case]:
    return all_cases()


@functools.lru_cache(maxsize=None)
def expected(i: int):
    c = cases()[i]
    return c.coded_list() if c.kind == "coded" else c.aux_list(c.frames)


def legacy_records(oracle_mod, c: Case) -> np.ndarray:
    """The records the engine must poll: the legacy oracle on every stream in (capture, channel) order."""
    out = []
    for cap in range(c.words.shape[0]):
        for ch in range(N_CH):
            if not c.words[cap, ch].any():
                continue
            b = np.unpackbits(c.words[cap, ch, 4:].view(np.uint8), bitorder="little")[: c.n_out]
            fr = oracle_mod.ble_decode(bb.bits_to_iq(b), ch)
            fr["channel"], fr["capture_id"] = ch, c.first_capture + cap
            out.append(fr)
    return np.concatenate(out) if out else np.zeros(0, _abi.FRAME_DTYPE)


def aux_against_records(c: Case, got, records):
    """The list on the engine's records equals the list on the synthetic records, but for depth-0 parents (the records of
    the aux packets on the data channels come first).  A record that two receiver windows both report (btle_rx's
    half-buffer overlap) is a second source of the same pointers: then only the sources are compared."""
    adv = records[(records["channel"] >= 37) & (records["proto"] == 3)]
    assert set(adv["sample_index"].tolist()) == set(c.frames["sample_index"].tolist()), c.name
    if len(adv) != len(c.frames):
        return
    want = c.aux_list(c.frames)
    assert len(got) == len(want)
    for k in want.dtype.names:
        if k != "parent":
            assert np.array_equal(got[k], want[k]), (c.name, k)
    d0 = got["depth"] == 0
    assert np.array_equal(records["sample_index"][got["parent"][d0]], c.frames["sample_index"][want["parent"][d0]]), c.name
    assert np.array_equal(got["parent"][~d0], want["parent"][~d0]), c.name


# ------------------------------------------------------------------------------------------------ CPU: every case means something
def test_every_case_fires_its_edge(oracle_mod):
    for i, c in enumerate(cases()):
        got = expected(i)
        c.check(got)
        if c.kind == "aux" and c.shard is None:
            rec = legacy_records(oracle_mod, c)
            for cap, ch, s in c.spots:
                assert ((rec["sample_index"] == s) & (rec["channel"] == ch) & (rec["crc_ok"] == 1)).any(), (c.name, s)
            aux_against_records(c, c.aux_list(rec), rec)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def Engine():
    from snout_b200.engine import RxEngine
    assert _abi.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return RxEngine


@pytest.fixture(scope="module")
def engine(Engine):
    n = max(c.n_out for c in cases())
    with Engine("ble_wb40", max_samples=24 * n, max_captures=3) as e:
        yield e


def run_case(e, c: Case):
    return e.run_bits(c.words, 24 * c.n_out, shard=c.shard_arg() if (c.shard or c.first_capture) else None)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["coded", "aux"])
def test_gpu_equals_oracles_on_every_case(engine, oracle_mod, kind):
    for i, c in enumerate(cases()):
        if c.kind != kind:
            continue
        rec = run_case(engine, c)
        if kind == "coded":
            assert_coded_equal(engine.ble_coded(), expected(i), c.name)
            continue
        for cap, ch, s in c.spots:
            assert ((rec["sample_index"] == s) & (rec["channel"] == ch) & (rec["crc_ok"] == 1)).any(), (c.name, s)
        if c.shard is None:
            assert_frames_equal(rec, legacy_records(oracle_mod, c), what=c.name)
        want = c.aux_list(rec)
        assert_aux_equal(engine.ble_aux(), want, c.name)
        if c.shard is None:
            aux_against_records(c, want, rec)


# ------------------------------------------------------------------------------------------------ A: the hook
@pytest.mark.gpu
def test_hook_round_trip_and_refusals(Engine):
    n_out = 5000
    nw = 4 + (n_out + 31) // 32 + 64
    rng = np.random.default_rng(1)
    w = np.zeros((3, N_CH, nw), np.uint32)
    b = rng.integers(0, 2, (3, N_CH, n_out), dtype=np.uint8)
    for cap in range(3):
        for ch in range(N_CH):
            w[cap, ch] = bb.pack_words(b[cap, ch], n_words=nw)
    with Engine("ble_wb40", max_samples=24 * n_out, max_captures=3) as e:
        e.run_bits(w, 24 * n_out)
        assert np.array_equal(e.debug_stage(_abi.STAGE_BLE_BITS), w)

        def code(words, n_samples, caps=None, shard=None):
            words = np.ascontiguousarray(words, np.uint32)
            sh = byref(_abi.Shard(*shard)) if shard else None
            return e.lib.snrx_debug_process_bits(e.handle, words.ctypes.data_as(c_void_p) if words.size else None,
                                                 caps or words.shape[0], n_samples, sh)
        assert code(np.zeros(0), 24 * n_out, caps=1) == -1                          # NULL words
        assert code(w, 24 * n_out - 1) == -1                                         # not a multiple of 24
        for cap, ch, word, bit in ((0, 0, 0, 0), (2, 39, 3, 31), (1, 5, 4 + n_out // 32, n_out % 32), (0, 7, nw - 1, 0)):
            bad = w.copy()
            bad[cap, ch, word] |= np.uint32(1 << bit)                                # lead word / sample n_out / tail
            assert code(bad, 24 * n_out) == -1, (cap, ch, word, bit)
        last = w.copy()
        last[0, 0, 4 + (n_out - 1) // 32] |= np.uint32(1 << ((n_out - 1) % 32))     # sample n_out - 1 is the stream's
        assert code(last, 24 * n_out) == 0
        e.poll()
        assert code(w, 24 * (n_out + 1)) == -5                                       # SNRX_ERANGE
        assert code(np.zeros((4, N_CH, nw)), 24 * n_out) == -5
        assert code(w, 24 * n_out, shard=(24 * 100, 0, 0, 0)) == -1                  # pre halo not a multiple of 128
        assert code(w, 24 * n_out) == 0 and code(w, 24 * n_out) == 0
        assert code(w, 24 * n_out) == -7                                             # SNRX_ESTATE: both lanes queued
        e.poll(); e.poll()
    for mode, kw in (("mixed_wb56", {}), ("zb_wb16", {}), ("ble_wb40", dict(keep_streams=True)),
                     ("ble_wb40", dict(rf_metrics=True))):
        with Engine(mode, max_samples=24 * n_out, **kw) as e:
            ww = np.zeros((1, e.n_ble or 40, nw), np.uint32)
            assert e.lib.snrx_debug_process_bits(e.handle, ww.ctypes.data_as(c_void_p), 1, 24 * n_out, None) == -1, (mode, kw)


@pytest.mark.gpu
def test_process_after_hook_batches_is_undisturbed(Engine):
    cap = synth.coded_adv_capture(seconds=0.15, seed=9700, esn0_db=25.0, n_events=4, max_chain=2)
    c = next(c for c in cases() if c.name == "coded three primaries, one packet")
    a = next(c for c in cases() if c.name == "aux chain of 5")
    n = max(len(cap.iq), 24 * max(c.n_out, a.n_out))
    with Engine("ble_wb40", max_samples=n) as e:
        fresh = (e.run(cap.iq), e.ble_aux(), e.ble_coded())
    with Engine("ble_wb40", max_samples=n) as e:
        run_case(e, c); e.ble_coded(); e.ble_aux()
        run_case(e, a); e.ble_aux(); e.ble_coded()
        after = (e.run(cap.iq), e.ble_aux(), e.ble_coded())
    for x, y in zip(fresh, after):
        assert x.tobytes() == y.tobytes()
    assert len(fresh[2]) > 0


# ------------------------------------------------------------------------------------------------ E: capacity
def _capacity_coded(n_prim_ptr: int, n_prim_plain: int):
    """Coded primaries (S=2: no false primaries), n_prim_ptr of them with an AuxPtr to one 1M packet each."""
    rng = np.random.default_rng(90 + n_prim_ptr)
    n = n_prim_ptr + n_prim_plain
    bt = zeroed(4000 + 8000 * n + 8000, 90, (37, 38, 39, 9))
    for j in range(n):
        s = 2000 + 8000 * j
        ptr = synth.aux_ptr_bytes(9, 1, 30, 20, 0) if j < n_prim_ptr else None
        plant(bt.b[37], s, coded_decisions(prim_pdu(rng, ptr), 37, 2))
        if ptr:
            lo, _ = ao.window(30, 20, 1)
            plant_stride(bt.b[9], s - 320 + 32 + lo + 30, aux_symbols(9, aux_pdu(rng, 16)), 4)
    return words_of([bt]), bt.n


def _capacity_aux(n_src: int, deep: int):
    """n_src ADV_EXT_INDs on channel 37, each pointing at a 2M packet (not a legacy record); `deep` of those point once
    more: n_src + deep entries from n_src records."""
    rng = np.random.default_rng(95 + 10 * n_src + deep)
    bt = Batch(40000, seed=95)
    for c in (9, 10):
        bt.b[c] &= 0
    for j in range(n_src):
        s = 1000 + 3000 * j
        a1 = s + 120 * 10 + 20
        a2 = a1 + 120 * 50 + 20
        ptr2 = synth.aux_ptr_bytes(10, 1, 30, 50, 1) if j < deep else None
        plant_stride(bt.b[9], a1, aux_symbols(9, aux_pdu(rng, 20, ptr2)), 2)
        if ptr2:
            plant_stride(bt.b[10], a2, aux_symbols(10, aux_pdu(rng, 20)), 2)
        bt.frames.append(primary_record(s, synth.aux_ptr_bytes(9, 1, 30, 10, 1)))
    return aux_case(f"capacity aux {n_src}/{deep}", bt, lambda got: None)


CAPACITY = 9                                  # max_frames of the capacity test
CODED_ROUNDS = ((0, 8), (0, 9), (4, 1), (3, 4))   # (primaries with a pointer, without): 9, 10 (primaries), 9, 10 (pointers)
AUX_ROUNDS = ((5, 4), (5, 5), (5, 4))             # 9, 10 (second pointer round), 9 entries from 5 records


@pytest.mark.gpu
def test_capacity_and_the_next_batch(Engine, oracle_mod):
    """Lists of exactly max_frames entries equal the oracle's; one more entry, from the primaries or from a pointer round,
    is SNRX_EOVERFLOW; the batch after an overflow is right again."""
    with Engine("ble_wb40", max_samples=24 * 90000, max_frames=CAPACITY) as e:
        for n_ptr, n_plain in CODED_ROUNDS:
            w, n_out = _capacity_coded(n_ptr, n_plain)
            e.run_bits(w, 24 * n_out)
            want = co.coded_list(w, n_out)
            if len(want) > CAPACITY:
                with pytest.raises(_abi.SnrxError) as ei:
                    e.ble_coded()
                assert ei.value.code == -6
            else:
                assert_coded_equal(e.ble_coded(), want, f"{n_ptr}/{n_plain}")
        for n_src, deep in AUX_ROUNDS:
            c = _capacity_aux(n_src, deep)
            rec = run_case(e, c)
            want = c.aux_list(rec)
            if len(want) > CAPACITY:
                with pytest.raises(_abi.SnrxError) as ei:
                    e.ble_aux()
                assert ei.value.code == -6
            else:
                assert_aux_equal(e.ble_aux(), want, "capacity aux")


def test_capacity_rounds_sit_on_the_edge(oracle_mod):
    """The capacity test's batches give exactly max_frames entries and one more, as intended."""
    sizes = []
    for n_ptr, n_plain in CODED_ROUNDS:
        w, n_out = _capacity_coded(n_ptr, n_plain)
        got = co.coded_list(w, n_out)
        sizes.append((len(got), int((got["depth"] == 0).sum())))
    assert sizes[0][0] == CAPACITY and sizes[1][0] == CAPACITY + 1 and sizes[1][1] == CAPACITY + 1
    assert sizes[2][0] == CAPACITY and sizes[3][0] == CAPACITY + 1 and sizes[3][1] <= CAPACITY
    for (n_src, deep), size in zip(AUX_ROUNDS, (CAPACITY, CAPACITY + 1, CAPACITY)):
        c = _capacity_aux(n_src, deep)
        rec = legacy_records(oracle_mod, c)
        got = c.aux_list(rec)
        assert len(got) == size and len(rec) <= CAPACITY and (got["status"] == ao.OK).all()


# ------------------------------------------------------------------------------------------------ F: the legacy back end
@pytest.mark.gpu
def test_legacy_back_end_across_40_streams(Engine, oracle_mod):
    """Dense, capture-end and window-edge streams on all 40 channels of one batch: per-channel whitening, the advertising
    length gate on 37..39 only, and the (capture, channel, window) order, against the legacy oracle per channel."""
    n_out = 3 * 8192 + 777
    nw = 4 + (n_out + 31) // 32 + 64
    for seed in range(2):
        w = np.zeros((2, N_CH, nw), np.uint32)
        want = []
        for cap in range(2):
            for ch in range(N_CH):
                kind = (ch + cap + seed) % 3
                if kind == 0:
                    _, par = bb.dense(1000 * seed + 40 * cap + ch, n_out, channel=ch, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
                elif kind == 1:
                    _, par = bb.window_edges(2000 * seed + 40 * cap + ch, 8192 * (1 + ch % 2) - 160 + 4 * ch + cap,
                                             channel=ch, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF, crc_init=0x555555)
                else:                                             # a frame cut 32 (1 + ch) samples or less before the end
                    rng = np.random.default_rng(3000 * seed + 40 * cap + ch)
                    _, par = bb.dense(3000 * seed + 40 * cap + ch, n_out, channel=ch, aa=bb.ADV_AA, aa_mask=0xFFFFFFFF,
                                      crc_init=0x555555)
                    bb.plant(par["bits"], n_out - 32 * (1 + ch) + int(rng.integers(-31, 1)),
                             bb.random_frame(rng, ch, bb.ADV_AA, 0x555555, length=int(rng.integers(6, 38)), crc_ok=True))
                b = np.zeros(n_out, np.uint8)
                m = min(n_out, len(par["bits"]))
                b[:m] = par["bits"][:m]
                b[n_out - 1] = 0
                w[cap, ch] = bb.pack_words(b, n_words=nw)
                fr = oracle_mod.ble_decode(bb.bits_to_iq(b), ch)
                fr["channel"], fr["capture_id"] = ch, cap
                want.append(fr)
        want = np.concatenate(want)
        with Engine("ble_wb40", max_samples=24 * n_out, max_captures=2) as e:
            got = e.run_bits(w, 24 * n_out)
        assert_frames_equal(got, want, what=f"seed {seed}")
        assert len(want) > 500 and len(set(want["channel"])) == N_CH


@pytest.mark.gpu
def test_candidate_capacity_across_channels(Engine):
    """Exactly 2^16 access-address candidates spread over the channels are taken; 2^16 + 1 overflow."""
    per = [1 << 16 >> 4] * 16
    n_out = 200 + 128 * (max(per) // 4 + 1) + 2000
    nw = 4 + (n_out + 31) // 32 + 64
    a = bb.aa_bits(bb.ADV_AA)
    for extra, over in ((0, False), (1, True)):
        w = np.zeros((1, N_CH, nw), np.uint32)
        total = 0
        for k, cnt in enumerate(per):
            ch = 2 * k + 1
            cnt = cnt + (extra if k == 0 else 0)
            b = np.zeros(n_out, np.uint8)
            for i in range(cnt):
                bb.plant(b, 200 + 128 * (i // 4) + (i % 4), a)
            total += bb.count_candidates(b, bb.ADV_AA, 0xFFFFFFFF)
            w[0, ch] = bb.pack_words(b, n_words=nw)
        assert total == (1 << 16) + extra
        with Engine("ble_wb40", max_samples=24 * n_out, max_frames=1 << 14) as e:     # candidate capacity 4 * 2^14
            if over:
                with pytest.raises(_abi.SnrxError) as ei:
                    e.run_bits(w, 24 * n_out)
                assert ei.value.code == -6
            else:
                e.run_bits(w, 24 * n_out)
                assert e.stats()["candidates"] == 1 << 16
