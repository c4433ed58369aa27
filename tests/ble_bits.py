"""Constructed BLE bit streams: int8 IQ whose slicer decisions are exactly a chosen bit stream.

The BLE back end (access-address search, decode, the window resolver) sees nothing but the slicer decisions
b[n] = (I[n]Q[n+1] - I[n+1]Q[n]) > 0.  A capture that walks the unit circle in quarter turns,

    x[0] = (64, 0),   x[n+1] = x[n] * (+j) if b[n] = 1 else x[n] * (-j),

has I[n]Q[n+1] - I[n+1]Q[n] = +-4096 at every n, so every slicer (btle_rx.c, the oracle, the narrow-band and the
harness slicer) decides exactly b[n].  As cf32 the same capture is q / 128 = +-0.5 or 0, which the narrow-band quantiser
(scale 128) maps back to the same int8 values.  The last sample of a capture pairs with the zero sample past its end, so
its decision is 0 whatever b says.

The frame construction uses synth.ble_whitening / synth.ble_crc24 (the definitions), not the oracle's tables, so that it is
independent of what it checks.  Plain numpy; no engine.
"""
from __future__ import annotations

import numpy as np

from snout_b200 import synth

SPS = 4
WINDOW = 8192
ADV_AA = 0x8E89BED6
_QUARTER = np.array([[64, 0], [0, 64], [-64, 0], [0, -64]], dtype=np.int8)     # 64 * j^k


def bits_to_iq(b) -> np.ndarray:
    """int8 [n, 2] capture whose decision at sample n < len(b) - 1 is b[n] (the last decision is 0)."""
    b = np.asarray(b, dtype=np.uint8)
    k = np.zeros(len(b), dtype=np.int64)
    if len(b) > 1:
        k[1:] = np.cumsum(2 * b[:-1].astype(np.int64) - 1)
    return _QUARTER[k & 3]


def decisions(iq) -> np.ndarray:
    """b[n] = I[n]Q[n+1] - I[n+1]Q[n] > 0 in int64, the sample past the end being zero."""
    q = np.asarray(iq, dtype=np.int64).reshape(-1, 2)
    nxt = np.vstack([q[1:], np.zeros((1, 2), np.int64)])
    return (q[:, 0] * nxt[:, 1] - nxt[:, 0] * q[:, 1] > 0).astype(np.uint8)


def check_iq(b, iq) -> None:
    """The construction's self-check: every cross product is +-4096 and its sign is b."""
    q = np.asarray(iq, dtype=np.int64).reshape(-1, 2)
    cross = q[:-1, 0] * q[1:, 1] - q[1:, 0] * q[:-1, 1]
    assert np.all(np.abs(cross) == 4096)
    want = np.asarray(b, dtype=np.uint8).copy()
    want[-1:] = 0
    assert np.array_equal(decisions(iq), want)


def effective_bits(b) -> np.ndarray:
    """What the slicers see for a constructed stream: b with the last decision 0."""
    e = np.asarray(b, dtype=np.uint8).copy()
    e[-1:] = 0
    return e


def pack_words(b, lead_words: int = 4, n_words: int | None = None) -> np.ndarray:
    """b in the back end's bit layout: bit (n & 31) of word lead_words + (n >> 5) is b[n]; zero lead and tail words."""
    b = np.asarray(b, dtype=np.uint8)
    body = (len(b) + 31) // 32
    n_words = lead_words + body if n_words is None else n_words
    out = np.zeros(n_words, dtype=np.uint32)
    padded = np.zeros(body * 32, dtype=np.uint8)
    padded[: len(b)] = b
    out[lead_words:lead_words + body] = np.packbits(padded, bitorder="little").view("<u4")
    return out


def lsb_bits(data) -> np.ndarray:
    return np.unpackbits(np.frombuffer(bytes(data), dtype=np.uint8), bitorder="little")


def aa_bits(aa: int) -> np.ndarray:
    return ((aa >> np.arange(32)) & 1).astype(np.uint8)


def plant(b: np.ndarray, s: int, symbols) -> None:
    """Write symbol-spaced bits b[s], b[s+4], ...; those outside the stream are dropped."""
    symbols = np.asarray(symbols, dtype=np.uint8)
    pos = s + SPS * np.arange(len(symbols))
    ok = (pos >= 0) & (pos < len(b))
    b[pos[ok]] = symbols[ok]


def crc_cmdline(init: int) -> int:
    """btle_rx's -k form of a CRCInit (its byte-swapped value), which the oracle and the engine take."""
    return ((init & 0xFF) << 16) | (init & 0xFF00) | ((init >> 16) & 0xFF)


def crc_internal(init: int) -> int:
    """crc_init_reorder(-k) of btle_rx: the CRCInit bit-reversed, the register the CRC starts from."""
    return int(f"{init & 0xFFFFFF:024b}"[::-1], 2)


def frame_symbols(channel: int, header: bytes, payload: bytes, crc_ok: bool = True, aa: int = ADV_AA,
                  crc_init: int = 0x555555, flip_aa_bits=()) -> np.ndarray:
    """Access address (LSB first) | whiten(header | payload | CRC-24) as symbols.  crc_ok=False flips one CRC bit."""
    pdu = bytes(header) + bytes(payload)
    crc = bytearray(synth.ble_crc24(pdu, crc_init))
    if not crc_ok:
        crc[1] ^= 0x10
    body = np.frombuffer(pdu + bytes(crc), dtype=np.uint8) ^ synth.ble_whitening(channel, len(pdu) + 3)
    a = aa_bits(aa)
    for k in flip_aa_bits:
        a[k] ^= 1
    return np.concatenate([a, lsb_bits(body.tobytes())])


def header_for(rng, channel: int, length: int) -> bytes:
    """A header whose length field is `length` (6 bits on advertising channels, 5 on data channels; the other bits random)."""
    b0 = int(rng.integers(0, 256))
    if 37 <= channel <= 39:
        b1 = (length & 0x3F) | (int(rng.integers(0, 4)) << 6)
    else:
        b1 = (length & 0x1F) | (int(rng.integers(0, 8)) << 5)
    return bytes([b0, b1])


def random_frame(rng, channel: int, aa: int, crc_init: int, length: int | None = None, crc_ok: bool | None = None,
                 flip_aa: bool = False) -> np.ndarray:
    """A frame with a length field of 0..63 (both sides of the advertising gate 6..37; data channels read 5 bits of it)."""
    if length is None:
        length = int(rng.integers(0, 64))
    if crc_ok is None:
        crc_ok = bool(rng.random() < 0.8)
    n_payload = length & (0x3F if 37 <= channel <= 39 else 0x1F)
    payload = rng.integers(0, 256, min(n_payload, 40), dtype=np.uint8).tobytes()
    flips = (int(rng.integers(0, 32)),) if flip_aa else ()
    return frame_symbols(channel, header_for(rng, channel, length), payload, crc_ok, aa, crc_init, flips)


# ------------------------------------------------------------------------------------------------ stream families

CHANNELS = (37, 38, 39, 0, 5, 36, 12)
AAS = (ADV_AA, 0x8E89BE00, 0x50000000, 0xA5A5A5A5)
MASKS = (0xFFFFFFFF, 0xFFFFFF00, 0xFFFF0000, 0x0000FFFF, 0xFFFFFFFE)


def _fill(rng, n: int) -> np.ndarray:
    return rng.integers(0, 2, n, dtype=np.uint8)


def _params(rng, channel=None, aa=None, aa_mask=None, crc_init=None) -> dict:
    ch = int(rng.choice(CHANNELS)) if channel is None else channel
    fixed_pair = aa is not None and aa_mask is not None
    if aa is None:
        aa = int(rng.choice(AAS)) if rng.random() < 0.6 else int(rng.integers(0, 1 << 32, dtype=np.uint64))
    if aa_mask is None:
        aa_mask = int(rng.choice(MASKS)) if rng.random() < 0.7 else int(rng.integers(0, 1 << 32, dtype=np.uint64))
    if crc_init is None:
        crc_init = 0x555555 if rng.random() < 0.4 else int(rng.integers(0, 1 << 24))
    if aa & aa_mask == 0 and not fixed_pair:      # no compared 1 bit: refused by the engine (DESIGN §4), pinned on its own
        aa, aa_mask = ADV_AA, 0xFFFFFFFF
    return dict(channel=ch, aa=aa, aa_mask=aa_mask, crc_init=crc_init)


def _finish(b, par) -> tuple[np.ndarray, dict]:
    par = dict(par, crc_cmdline=crc_cmdline(par["crc_init"]))
    return bits_to_iq(b), dict(par, bits=effective_bits(b))


def dense(seed: int, n: int | None = None, **fixed):
    """Frames every 20..700 samples at all four phases, lengths 0..63, right and wrong CRCs, 30 % with one access-address bit
    flipped, over random fill."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    n = int(rng.integers(1_000, 41_000)) if n is None else n
    b = _fill(rng, n)
    s = int(rng.integers(-100, 300))
    while s < n:
        plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"], flip_aa=rng.random() < 0.3))
        s += int(rng.integers(20, 701))
    return _finish(b, par)


def near_misses(seed: int, **fixed):
    """True copies of the access address next to copies with one or two flipped bits and copies shifted by one sample."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    n = int(rng.integers(8_000, 30_000))
    b = _fill(rng, n)
    s = int(rng.integers(0, 200))
    while s < n:
        kind = int(rng.integers(0, 4))
        f = random_frame(rng, par["channel"], par["aa"], par["crc_init"], crc_ok=True)
        if kind == 1:
            f[rng.choice(32, 1 + int(rng.integers(0, 2)), replace=False)] ^= 1
        plant(b, s, f)
        if kind == 2:                                             # the same address one sample later or earlier
            plant(b, s + int(rng.choice([-1, 1])), aa_bits(par["aa"]))
        elif kind == 3:                                           # a one-bit miss just before a true copy
            a = aa_bits(par["aa"]); a[int(rng.integers(0, 32))] ^= 1
            plant(b, s - int(rng.integers(1, 8)), a)
        s += int(rng.integers(150, 900))
    return _finish(b, par)


def lookalikes(seed: int, **fixed):
    """Frames whose payload carries a copy of the access address, symbol-aligned and misaligned: the receiver resumes after
    the frame and must not report the copy."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    ch, aa = par["channel"], par["aa"]
    n = int(rng.integers(8_000, 30_000))
    b = _fill(rng, n)
    s = int(rng.integers(0, 200))
    while s < n:
        length = int(rng.integers(8, 38))
        f = random_frame(rng, ch, aa, par["crc_init"], length=length, crc_ok=True)
        plant(b, s, f)
        at = s + 4 * (32 + 16 + int(rng.integers(0, 8 * (length - 4))))   # a symbol of the payload
        plant(b, at + int(rng.choice([0, 0, 1, 2, 3])), aa_bits(aa))
        s += 4 * len(f) + int(rng.integers(20, 400))
    return _finish(b, par)


def window_edges(seed: int, off: int, **fixed):
    """Access-address bit 0 at sample `off` (the tests take every offset in [8192k - 160, 8192k + 8]), with frames before and
    after it: the earlier ones make the search of window k - 1 reach `off` with every amount of eaten input, so that headers
    and payloads also cross the demodulation limit (19392 int8 past the window start)."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    n = WINDOW * (off // WINDOW + 2) + int(rng.integers(0, 3000))
    b = _fill(rng, n)
    s = max(off - 4 * 32 * int(rng.integers(0, 30)), -64)       # earlier frames first, the one at `off` last
    while s < off:
        plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"]))
        s += int(rng.integers(300, 700))
    plant(b, off, random_frame(rng, par["channel"], par["aa"], par["crc_init"], crc_ok=True))
    s = off + int(rng.integers(200, 800))
    while s < n:
        plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"]))
        s += int(rng.integers(20, 700))
    return _finish(b, dict(par, edge=off))


def capture_end(seed: int, cut_words: int, **fixed):
    """A frame starts 32 * cut_words samples (plus a random phase) before the capture ends."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    n0 = int(rng.integers(0, 3 * WINDOW))
    n = n0 + 32 * cut_words + int(rng.integers(-31, 1))
    n = max(n, 1)
    b = _fill(rng, n)
    s = int(rng.integers(0, 400))
    while s < n0 - 1500:
        plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"]))
        s += int(rng.integers(20, 700))
    plant(b, n0, random_frame(rng, par["channel"], par["aa"], par["crc_init"], length=int(rng.integers(6, 38)), crc_ok=True))
    return _finish(b, dict(par, start=n0))


def short(seed: int, n: int, **fixed):
    """A capture of exactly n samples (n of any residue, shorter than a window too) filled with frames."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    b = _fill(rng, n)
    s = int(rng.integers(-120, 60))
    while s < n:
        plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"]))
        s += int(rng.integers(20, 500))
    return _finish(b, par)


def virtual_aa(rng, z: int) -> tuple[int, int]:
    """(aa, mask) such that aa & mask has exactly z trailing zeros (0 <= z <= 31)."""
    mask = (int(rng.integers(0, 1 << 32, dtype=np.uint64)) | (1 << z)) if rng.random() < 0.5 else 0xFFFFFFFF
    aa = int(rng.integers(0, 1 << 32, dtype=np.uint64))
    aa = ((aa >> (z + 1)) << (z + 1)) | (1 << z)
    return aa & 0xFFFFFFFF, mask


def virtual_history(seed: int, z: int, **fixed):
    """An address whose masked low z bits are zero (aa & mask has z trailing zeros, 0 <= z <= 31).  With such an address a
    zeroed history matches the first z positions, so a frame can be found up to z symbols before a search origin.  Frames
    are planted around the origins that the stream makes: window starts and the points where the search resumes after a
    frame or after a header that fails the advertising length gate."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    if "aa" not in fixed:
        aa, mask = virtual_aa(rng, z)
        par.update(aa=aa, aa_mask=mask)
    ch, aa = par["channel"], par["aa"]
    n = int(rng.integers(2 * WINDOW, 4 * WINDOW))
    b = _fill(rng, n)
    s = int(rng.integers(-124, 4))
    while s < n:
        adv = 37 <= ch <= 39
        length = int(rng.choice([3, 50])) if adv and rng.random() < 0.3 else int(rng.integers(0, 38))
        f = random_frame(rng, ch, aa, par["crc_init"], length=length)
        plant(b, s, f)
        gated = adv and not 6 <= length <= 37
        end = s + 4 * (32 + 16 + (0 if gated else 8 * ((length & (0x3F if adv else 0x1F)) + 3)))
        s = end + 4 * int(rng.integers(0, 32)) + int(rng.integers(0, 4)) - 4 * int(rng.integers(0, z + 1))
        if rng.random() < 0.15:                                  # next window start
            s = (s // WINDOW + 1) * WINDOW + 4 * int(rng.integers(0, 32)) - 4 * min(z, 31)
    return _finish(b, par)


def pathological(seed: int, kind: str, **fixed):
    """All zeros, all ones, 0x55 / 0xAA preambles, and fill in which every lane of the bit-parallel correlation survives
    past position 11 (the address itself at every fourth sample, with one flipped bit past position 11)."""
    rng = np.random.default_rng(seed)
    par = _params(rng, **fixed)
    n = int(rng.integers(9_000, 20_000))
    if kind == "zeros":
        b = np.zeros(n, np.uint8)
    elif kind == "ones":
        b = np.ones(n, np.uint8)
    elif kind in ("x55", "xaa"):
        b = np.tile(lsb_bits(bytes([0x55 if kind == "x55" else 0xAA])), n // 8 + 1)[:n].copy()
        s = int(rng.integers(0, 300))
        while s < n:
            plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"]))
            s += int(rng.integers(400, 1200))
    elif kind == "survivors":
        a = aa_bits(par["aa"])
        b = np.zeros(n, np.uint8)
        for ph in range(4):                                       # every phase is the address, repeated, with a late miss
            rep = np.tile(a, n // 128 + 2)
            rep[12 + 32 * np.arange(n // 128 + 2) + ph % 4] ^= 1
            b[ph::4] = rep[: len(b[ph::4])]
        s = int(rng.integers(0, 300))
        while s < n:
            plant(b, s, random_frame(rng, par["channel"], par["aa"], par["crc_init"], crc_ok=True))
            s += int(rng.integers(600, 1500))
    else:
        raise ValueError(kind)
    return _finish(b, par)


def capacity_stream(n_cands: int, seed: int = 0, aa: int = ADV_AA, n_frames: int = 24) -> np.ndarray:
    """n_cands copies of the address: n_cands - n_frames bare ones back to back at the four phases in turn (four per 128
    samples), then n_frames advertising frames with a correct CRC, over random fill.  count_candidates() says how many
    positions match in all."""
    rng = np.random.default_rng(seed)
    bare = n_cands - n_frames
    body = 200 + 32 * bare + 128
    n = body + 800 * n_frames + 1000
    b = _fill(rng, n)
    a = aa_bits(aa)
    for i in range(bare):
        plant(b, 200 + 128 * (i // 4) + (i % 4), a)
    for i in range(n_frames):
        plant(b, body + 800 * i + i % 4, random_frame(rng, 37, aa, 0x555555, length=int(rng.integers(6, 38)), crc_ok=True))
    return b


def count_candidates(b, aa: int, mask_hi: int) -> int:
    """Start positions s in [-128, n) -- the ones the correlation has words for -- where every position of mask_hi matches
    the address (samples outside the capture are zero).  mask_hi: the compared positions above the virtual ones,
    mask & ~((1 << z) - 1) with z the trailing zeros of aa & mask."""
    b = np.asarray(b, dtype=np.uint8)
    n = len(b)
    ext = np.concatenate([np.zeros(128, np.uint8), b, np.zeros(128, np.uint8)])
    ok = np.ones(n + 128, dtype=bool)
    for p in range(32):
        if (mask_hi >> p) & 1:
            ok &= ext[4 * p:4 * p + n + 128] == ((aa >> p) & 1)
    return int(ok.sum())


def mask_hi(aa: int, mask: int) -> int:
    v = aa & mask
    z = min((v & -v).bit_length() - 1, 31) if v else 31
    return mask & ~((1 << z) - 1) & 0xFFFFFFFF
