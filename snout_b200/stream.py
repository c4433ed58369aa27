"""Streaming front door of the receive engine: an unbounded IQ stream cut into time shards.

`btle_rx` consumes an endless HackRF stream half buffer by half buffer
(vendor/BTLE/host/btle-tools/src/btle_rx.c:2341-2393) and the Zigbee flowgraph runs until it is told
to stop (snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py:121-126).  The CUDA engine works on
batches, so the stream is cut into shards on the grids the results are defined on (8192-sample
BLE windows, Zigbee segments) with the halos of include/snoutrx.h `snrx_shard_t`; by construction
the frames are those of one call over the whole stream, bit for bit (tests/test_gpu_parity.py
*_shards_equal_whole, tests/test_stream.py).

Two shards are kept in flight (process k+1 is queued before k is collected) and the shard
buffers are page-locked, so host->device copies overlap the kernels.
"""
from __future__ import annotations

import os
from typing import BinaryIO, Iterator

import numpy as np

from . import _abi, chanplan

ZB_IIR_MEMORY = (_abi.ZB_IIR_MEMORY_BLOCKS + 1) * _abi.ZB_IIR_BLOCK    # the remembered blocks + the buffer's first block (include/snoutrx.h)
ZB_POST_HALO = 16448 + 64         # kZbPostHalo (csrc/zb.cuh) rounded up
BLE_PRE_HALO = 128
BLE_POST_HALO = 2048


def shard_geometry(n_ble: int, n_zb: int, zb_segment: int = 0, zb_prehalo: int = 0) -> tuple[int, int, int]:
    """(unit, pre, post) in channel-rate samples for an engine with n_ble / n_zb receivers (0 = the library defaults)."""
    zb_segment = zb_segment or _abi.ZB_SEGMENT_DEFAULT
    zb_prehalo = zb_prehalo or _abi.ZB_PREHALO_DEFAULT
    unit, pre, post = chanplan.BLE_WINDOW, 0, 0
    if n_ble:
        pre, post = BLE_PRE_HALO, BLE_POST_HALO
    if n_zb:
        if zb_segment % chanplan.BLE_WINDOW and chanplan.BLE_WINDOW % zb_segment:
            raise ValueError("zb_segment must divide 8192 or be a multiple of it for sharded operation")
        unit = max(zb_segment, chanplan.BLE_WINDOW)      # shard bodies start on the 8192-sample window grid
        need = ZB_IIR_MEMORY + zb_prehalo
        pre = max(pre, -(-need // _abi.ZB_IIR_BLOCK) * _abi.ZB_IIR_BLOCK)
        post = max(post, ZB_POST_HALO)
    return unit, pre, post


def plan_shards(n_samples: int, decim: int, unit: int, pre: int, post: int, units_per_shard: int) -> list[dict]:
    """Cut a capture of n_samples input-rate samples into shards: list of
    {lo, hi, pre_samples, body_samples, first_window} (input-rate samples; first_window in 8192 windows)."""
    n_ch = n_samples // decim
    body = unit * units_per_shard
    out = []
    b0 = 0
    while b0 < n_ch or not out:
        b1 = min(n_ch, b0 + body)
        lo = max(0, b0 - pre)
        hi = min(n_ch, b1 + post)
        last = b0 + body + post >= n_ch            # the stream ends inside this shard's post halo: take the rest
        out.append(dict(lo=lo * decim, hi=(n_ch if last else hi) * decim, pre_samples=(b0 - lo) * decim,
                        body_samples=0 if last else (b1 - b0) * decim, first_window=b0 // chanplan.BLE_WINDOW))
        if last:
            break
        b0 = b1
    return out


def zb_span_filter(frames: np.ndarray, state: dict | None = None) -> np.ndarray:
    """The 802.15.4 span rule across shard boundaries (include/snoutrx.h, csrc/zb.cuh k_zb_span_filter): a CRC-failed
    record whose sync lies inside the span of an earlier CRC-ok record of the same (capture, channel) stream is dropped.
    The engine applies the rule inside a batch; the CRC-ok frame that covers the first records of a time shard was
    reported by the previous shard, so whoever concatenates shards applies it once more.  `frames`: records in stream
    order per (capture, channel) (any interleaving of streams); `state` carries the end of the last CRC-ok frame of
    every stream from call to call (streaming).  Idempotent; BLE records pass through."""
    if len(frames) == 0:
        return frames
    zb = frames["proto"] == 2
    if not zb.any():
        return frames
    keep = np.ones(len(frames), dtype=bool)
    key = frames["capture_id"].astype(np.int64) * 65536 + frames["channel"].astype(np.int64)
    ends = frames["sample_index"] + (2 + 2 * frames["len"].astype(np.int64)) * 64
    for k in np.unique(key[zb]):
        idx = np.nonzero(zb & (key == k))[0]
        s = frames["sample_index"][idx]
        ok = frames["crc_ok"][idx] == 1
        e = np.where(ok, ends[idx], 0)
        prev = state.get(int(k), 0) if state is not None else 0
        before = np.maximum.accumulate(np.concatenate(([prev], e)))[:-1]      # end of the CRC-ok frames seen so far
        keep[idx] = ok | (s >= before)
        if state is not None:
            state[int(k)] = int(max(prev, e.max()))
    return frames if keep.all() else frames[keep]


def rf_of(frames: np.ndarray, rf: np.ndarray) -> np.ndarray:
    """The radio-metrics records (RxEngine.frame_rf()) of `frames`, matched on their key fields (capture, sample index,
    channel, protocol): the streamer filters and a caller may reorder the records of a batch.  A frame without a match gets
    a record whose valid bits are clear."""
    from ._abi import RF_DTYPE
    out = np.zeros(len(frames), dtype=RF_DTYPE)
    out[["power_dbfs", "noise_dbfs", "snr_db", "cfo_hz"]] = (np.nan, np.nan, np.nan, np.nan)
    index = {(int(r["capture_id"]), int(r["sample_index"]), int(r["channel"]), int(r["proto"])): i for i, r in enumerate(rf)}
    for i, f in enumerate(frames):
        j = index.get((int(f["capture_id"]), int(f["sample_index"]), int(f["channel"]), int(f["proto"])))
        if j is not None:
            out[i] = rf[j]
    return out


class ShardStreamer:
    """Push IQ blocks in, get frame arrays out, in stream order.

        st = ShardStreamer(engine)
        for block in blocks:             # complex64 numpy arrays of any length
            for frames in st.feed(block): ...
        for frames in st.flush(): ...
    """

    def __init__(self, engine, units_per_shard: int | None = None):
        self.eng = engine
        self.decim = engine.decim
        self.unit, self.pre, self.post = shard_geometry(engine.n_ble, engine.n_zb, engine.cfg.zb_segment, engine.cfg.zb_prehalo)
        cap_in = int(engine.cfg.max_samples) or (96_000_000 if engine.wideband else 10_000_000)   # snrx_create defaults
        cap_ch = cap_in // self.decim
        room = (cap_ch - self.pre - self.post) // self.unit
        if room < 1:
            raise ValueError(f"engine max_samples too small for one shard: need >= {(self.unit + self.pre + self.post) * self.decim}")
        self.units = min(room, units_per_shard) if units_per_shard else room
        self.body = self.units * self.unit
        self.cap_in = (self.pre + self.body + self.post) * self.decim
        self.slots = [engine.alloc_host(self.cap_in) for _ in range(2)]      # page-locked (snrx_host_alloc)
        self.cur = 0                     # slot being filled
        self.fill = 0                    # input-rate samples in the slot
        self.body_start = 0              # channel-rate index of the body of the shard being filled
        self.in_flight = 0
        self.total_in = 0
        self._zb_state = {}              # zb_span_filter state: the shards of a stream come back in order

    def _poll(self) -> np.ndarray:
        fr = self.eng.poll()
        return zb_span_filter(fr, self._zb_state) if self.eng.n_zb else fr

    # absolute input-rate index of the first sample of the slot being filled
    def _lo(self) -> int:
        return max(0, self.body_start - self.pre) * self.decim

    def _target(self) -> int:
        return (self.body_start + self.body + self.post) * self.decim - self._lo()

    def _launch(self, last: bool) -> None:
        slot = self.slots[self.cur].array
        lo = self._lo()
        n = self.fill
        if self.decim > 1:
            n -= n % self.decim
        shard = dict(pre_samples=self.body_start * self.decim - lo, body_samples=0 if last else self.body * self.decim,
                     first_window=self.body_start // chanplan.BLE_WINDOW)
        self.eng.process(slot[:n], shard=shard)
        self.in_flight += 1

    def _advance(self) -> None:
        """After launching the shard in slot `cur`: seed the other slot with the overlap."""
        src = self.slots[self.cur].array
        old_lo = self._lo()
        self.body_start += self.body
        new_lo = self._lo()
        keep = old_lo + self.fill - new_lo
        other = self.slots[self.cur ^ 1].array
        other[:keep] = src[new_lo - old_lo: new_lo - old_lo + keep]
        self.cur ^= 1
        self.fill = keep

    def feed(self, block: np.ndarray) -> Iterator[np.ndarray]:
        block = np.asarray(block, dtype=np.complex64).reshape(-1)
        self.total_in += len(block)
        off = 0
        while off < len(block):
            slot = self.slots[self.cur].array
            take = min(len(block) - off, self._target() - self.fill)
            slot[self.fill: self.fill + take] = block[off: off + take]
            self.fill += take
            off += take
            if self.fill == self._target():
                if self.in_flight == 2:              # the slot we are about to seed belongs to the oldest batch
                    yield self._poll()
                    self.in_flight -= 1
                self._launch(last=False)
                if self.in_flight == 2:
                    yield self._poll()
                    self.in_flight -= 1
                self._advance()

    def flush(self) -> Iterator[np.ndarray]:
        """End of stream: the remaining samples form the last shard."""
        n_eff = self.fill - self.fill % self.decim
        if n_eff > self.body_start * self.decim - self._lo():          # anything past the pre halo
            if self.in_flight == 2:
                yield self._poll()
                self.in_flight -= 1
            self._launch(last=True)
        while self.in_flight:
            yield self._poll()
            self.in_flight -= 1
        self.fill = 0

    def close(self):
        for s in self.slots:
            s.free()
        self.slots = []


# ---------------------------------------------------------------------------------- IQ sources
def iq_blocks(source: str | BinaryIO, fmt: str = "cf32", block_samples: int = 1 << 22, scale: float | None = None
              ) -> Iterator[np.ndarray]:
    """Read interleaved IQ from a file, '-' (stdin) or a binary file object and yield complex64 blocks.

    fmt  cf32  interleaved float32 (GNU Radio file sink, the BASELINE capture format)
         sc8   interleaved int8 as the HackRF delivers it to btle_rx (rx_callback, btle_rx.c:489-498);
               values become q / scale (default 128) so the engine's quantiser restores q exactly
    """
    fh = source
    close = False
    if isinstance(source, str):
        if source == "-":
            fh = os.fdopen(0, "rb", closefd=False)
        else:
            fh = open(source, "rb")
            close = True
    try:
        item = 8 if fmt == "cf32" else 2
        while True:
            raw = fh.read(block_samples * item)
            if not raw:
                break
            raw = raw[: len(raw) - len(raw) % item]
            if fmt == "cf32":
                yield np.frombuffer(raw, dtype=np.complex64)
            elif fmt == "sc8":
                q = np.frombuffer(raw, dtype=np.int8).astype(np.float32) * np.float32(1.0 / (scale or 128.0))
                yield q.view(np.complex64)
            else:
                raise ValueError(f"unknown IQ format {fmt}")
    finally:
        if close:
            fh.close()
