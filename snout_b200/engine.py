"""RxEngine -- Python host of the receive engine (thin layer over the C ABI).

Mirrors the two receiver interfaces of Snout on the hot path:

* BLE: what `btle_rx -c <ch> -a <aa> -k <crcinit>` does per channel
  (vendor/BTLE/host/btle-tools/src/btle_rx.c:2288-2393), here for one channel (narrow band) or all
  40 at once (wideband);
* Zigbee: what the flowgraph `top_block(channel=...)` does
  (snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py:29-103), one channel or all 16.

All DSP runs in libsnoutrx.so on the GPU.  This module only moves pointers and records.
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_uint32, c_uint64, c_void_p

import numpy as np

from . import _abi, chanplan
from ._abi import (FRAME_DTYPE, MODE_BLE_NB, MODE_BLE_WB40, MODE_MIXED_WB56, MODE_ZB_NB, MODE_ZB_WB16, Config, Shard,
                   SnrxError, Stats)

MODES = {
    "ble_nb": MODE_BLE_NB, "zb_nb": MODE_ZB_NB, "zb_wb16": MODE_ZB_WB16, "ble_wb40": MODE_BLE_WB40,
    "mixed_wb56": MODE_MIXED_WB56,
}


def _is_torch_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


class RxEngine:
    """One engine = one GPU + one receive mode.  Not thread safe; engines are independent."""

    def __init__(self, mode: str | int = "ble_nb", channel: int | None = None, device: int = 0,
                 max_samples: int = 0, max_captures: int = 1, max_frames: int = 0,
                 access_addr: int = chanplan.BLE_ADV_AA, crc_init: int = chanplan.BLE_ADV_CRC_INIT,
                 zb_threshold: int = 10, quant_scale: float = 0.0, zb_segment: int = 0, zb_prehalo: int = 0,
                 pfb_taps: int = 0, keep_streams: bool = False, access_mask: int = 0, rf_metrics: bool = False):
        self.lib = _abi.load()
        self.mode = MODES[mode] if isinstance(mode, str) else int(mode)
        if channel is None:
            channel = 11 if self.mode == MODE_ZB_NB else 37
        cfg = Config()
        cfg.abi_version = _abi.ABI_VERSION
        cfg.device = device
        cfg.mode = self.mode
        cfg.channel = channel
        cfg.access_addr = access_addr
        cfg.crc_init = crc_init
        cfg.zb_threshold = zb_threshold
        cfg.quant_scale = quant_scale
        cfg.max_samples = max_samples
        cfg.max_captures = max_captures
        cfg.max_frames = max_frames
        cfg.zb_segment = zb_segment
        cfg.zb_prehalo = zb_prehalo
        cfg.pfb_taps = pfb_taps
        cfg.flags = (_abi.F_KEEP_STREAMS if keep_streams else 0) | (_abi.F_RF_METRICS if rf_metrics else 0)
        cfg.access_mask = access_mask & 0xFFFFFFFF
        self.cfg = cfg
        self.max_frames = int(cfg.max_frames) or (1 << 17)     # records per batch; 1 << 17: the library default
        self.handle = c_void_p()
        rc = self.lib.snrx_create(byref(self.handle), byref(cfg))
        if rc != 0:
            what = self.lib.snrx_strerror(rc).decode()
            detail = self.lib.snrx_last_error(None).decode()
            self.handle = c_void_p()
            raise SnrxError(rc, what, detail)
        self.wideband = self.mode in (MODE_ZB_WB16, MODE_BLE_WB40, MODE_MIXED_WB56)
        self.decim = chanplan.WB_DECIM if self.wideband else 1
        self.n_ble = {MODE_BLE_NB: 1, MODE_BLE_WB40: 40, MODE_MIXED_WB56: 40}.get(self.mode, 0)
        self.n_zb = {MODE_ZB_NB: 1, MODE_ZB_WB16: 16, MODE_MIXED_WB56: 16}.get(self.mode, 0)
        self._keepalive = []             # inputs of the (up to two) batches in flight: released when their batch is polled
        self._last = None
        self.batches_queued = 0          # snrx_process calls so far = the number the library gives the next batch
        self.polled_batch_no = -1        # number of the batch most recently returned by poll()

    # ------------------------------------------------------------------ life cycle
    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.snrx_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise SnrxError(rc, self.lib.snrx_strerror(rc).decode(), self.lib.snrx_last_error(self.handle).decode())

    def _polled_list(self, fn, dtype, *args) -> np.ndarray:
        """A list about the batch most recently returned by poll(): fn(handle, *args, out, cap, &n) of the C ABI, with
        room for max_frames entries."""
        n = c_uint32(0)
        out = np.zeros(self.max_frames, dtype=dtype)
        self._check(fn(self.handle, *args, out.ctypes.data_as(c_void_p), self.max_frames, byref(n)))
        return out[: n.value].copy()

    # ------------------------------------------------------------------ control
    def set_channel(self, channel: int):
        """Narrow-band modes: retune (top_block.set_channel, top_block.py:94-96 / btle_rx -c)."""
        self._check(self.lib.snrx_set_channel(self.handle, int(channel)))

    def set_stream(self, cuda_stream: int | None):
        self._check(self.lib.snrx_set_stream(self.handle, c_void_p(cuda_stream or 0)))

    def sync(self):
        self._check(self.lib.snrx_sync(self.handle))

    # ------------------------------------------------------------------ data path
    def process(self, iq, shard: dict | None = None, n_samples: int | None = None, stride: int = 0):
        """Queue one batch.  `iq`: complex64 numpy array [n] or [captures, n] (host memory), a
        _abi.PinnedBuffer, or a torch CUDA tensor of complex64 [n] / [captures, n].  int8 arrays / tensors
        with a trailing axis of 2 ([n, 2] or [captures, n, 2]: interleaved I,Q as a HackRF delivers them,
        btle_rx.c:489-498) take the sc8 entry point; their sample value is q / 128.  The engine reads the input
        asynchronously (kernels on its own streams, chunked host->device copies): it keeps a reference until the batch has
        been polled; callers that pass raw pointers (process_device_ptr) must keep the memory alive themselves."""
        sh = None
        if shard:
            sh = Shard(int(shard.get("pre_samples", 0)), int(shard.get("body_samples", 0)),
                       int(shard.get("first_window", 0)), int(shard.get("first_capture_id", 0)))
        if isinstance(iq, _abi.PinnedBuffer):
            iq = iq.array
        if _is_torch_tensor(iq):
            import torch
            if not iq.is_cuda:
                iq = iq.numpy()
            else:
                assert iq.is_contiguous()
                if iq.dtype == torch.int8:
                    assert iq.shape[-1] == 2, "sc8 input is [..., n, 2] (I, Q)"
                    fn, shape = self.lib.snrx_process_sc8, iq.shape[:-1]
                else:
                    assert iq.dtype == torch.complex64
                    fn, shape = self.lib.snrx_process, iq.shape
                caps = 1 if len(shape) == 1 else shape[0]
                n = shape[-1] if n_samples is None else n_samples
                st = stride or shape[-1]
                self.set_stream(torch.cuda.current_stream(iq.device).cuda_stream)
                self._keepalive.append(iq)
                self._check(fn(self.handle, c_void_p(iq.data_ptr()), caps, n, st, byref(sh) if sh else None, 1))
                self._last = (caps, n)
                self.batches_queued += 1
                return self
        a = np.asarray(iq)
        if a.dtype == np.int8:
            if a.shape[-1] != 2:
                raise ValueError("sc8 input is [..., n, 2] (I, Q)")
            a = np.ascontiguousarray(a)
            fn, shape = self.lib.snrx_process_sc8, a.shape[:-1]
        else:
            if a.dtype != np.complex64 or not a.flags.c_contiguous:
                a = np.ascontiguousarray(a, dtype=np.complex64)
            fn, shape = self.lib.snrx_process, a.shape
        caps = 1 if len(shape) == 1 else shape[0]
        n = shape[-1] if n_samples is None else n_samples
        st = stride or shape[-1]
        self._keepalive.append(a)
        self._check(fn(self.handle, a.ctypes.data_as(c_void_p), caps, n, st, byref(sh) if sh else None, 0))
        self._last = (caps, n)
        self.batches_queued += 1
        return self

    def process_device_ptr(self, ptr: int, n_captures: int, n_samples: int, stride: int = 0, shard: Shard | None = None):
        self._check(self.lib.snrx_process(self.handle, c_void_p(ptr), n_captures, n_samples, stride,
                                          byref(shard) if shard else None, 1))
        self._last = (n_captures, n_samples)
        self.batches_queued += 1
        return self

    def process_bits(self, words, n_samples: int, shard: dict | None = None):
        """Test hook (snrx_debug_process_bits): queue a batch whose BLE slicer bit streams are `words` -- uint32
        [captures, BLE channels, words] in the SNRX_STAGE_BLE_BITS layout, for n_samples input samples per capture --
        instead of channelizing a capture.  poll() and every call on the polled batch then see these streams."""
        sh = None
        if shard:
            sh = Shard(int(shard.get("pre_samples", 0)), int(shard.get("body_samples", 0)),
                       int(shard.get("first_window", 0)), int(shard.get("first_capture_id", 0)))
        w = np.ascontiguousarray(words, dtype=np.uint32)
        caps = 1 if w.ndim < 3 else w.shape[0]
        self._check(self.lib.snrx_debug_process_bits(self.handle, w.ctypes.data_as(c_void_p), caps, int(n_samples),
                                                     byref(sh) if sh else None))
        self._keepalive.append(w)
        self._last = (caps, int(n_samples))
        self.batches_queued += 1
        return self

    def run_bits(self, words, n_samples: int, **kw) -> np.ndarray:
        return self.process_bits(words, n_samples, **kw).poll()

    def poll(self, copy: bool = True) -> np.ndarray:
        """Wait for the oldest queued batch (up to two may be queued) and return its frames in
        reference order (capture, channel, window, index).  copy=False returns a view of the engine's
        pinned result buffer, valid until the second-next process()."""
        n = c_uint32(0)
        ptr = c_void_p()
        try:
            self._check(self.lib.snrx_poll_view(self.handle, byref(ptr), byref(n)))
        finally:
            if self._keepalive:              # the oldest batch is done with its input (host copies and kernels have finished)
                self._keepalive.pop(0)
            self.polled_batch_no += 1
        if n.value == 0:
            return np.zeros(0, dtype=FRAME_DTYPE)
        buf = (ctypes.c_char * (n.value * FRAME_DTYPE.itemsize)).from_address(ptr.value)
        view = np.frombuffer(buf, dtype=FRAME_DTYPE)
        return view.copy() if copy else view

    def run(self, iq, **kw) -> np.ndarray:
        return self.process(iq, **kw).poll()

    def alloc_host(self, n_samples: int, sc8: bool = False) -> _abi.PinnedBuffer:
        """Page-locked staging buffer (snrx_host_alloc) for full-rate host->device copies: complex64 [n], or
        int8 [n, 2] with sc8=True."""
        if sc8:
            return _abi.PinnedBuffer((int(n_samples), 2), np.int8)
        return _abi.PinnedBuffer(int(n_samples), np.complex64)

    def stats(self) -> dict:
        s = Stats()
        self._check(self.lib.snrx_stats(self.handle, byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def polled_frames_device(self) -> tuple[int, int, int]:
        """(device address, capacity in records, count) of the frame list of the batch most recently returned by
        poll(): the HBM list the kernels wrote, valid for two further process() calls -- what dist.FrameGather
        sends over NVLink."""
        f, n = c_void_p(), c_uint32(0)
        self._check(self.lib.snrx_polled_frames_device(self.handle, byref(f), byref(n)))
        return int(f.value or 0), self.max_frames, int(n.value)

    # ------------------------------------------------------------------ SURVEY 8(e): frame exchange between engines
    def exchange_create(self, rank: int, world: int, cap_records: int = 1 << 15) -> bytes:
        """Allocate this engine's receive area; returns its 64-byte CUDA IPC handle (include/snoutrx.h snrx_exchange_create)."""
        buf = ctypes.create_string_buffer(_abi.XCHG_HANDLE_BYTES)
        self._check(self.lib.snrx_exchange_create(self.handle, rank, world, cap_records, buf))
        self._xchg_world = world
        return buf.raw

    def exchange_connect(self, handles: bytes):
        """`handles`: the handles of all ranks, concatenated in rank order.  Every batch queued afterwards is pushed to every
        rank by the kernel that exports it."""
        assert len(handles) == _abi.XCHG_HANDLE_BYTES * self._xchg_world
        self._check(self.lib.snrx_exchange_connect(self.handle, ctypes.c_char_p(handles)))

    def allgather(self, batch_no: int, want_frames: bool = False, timeout_ms: int = 30000):
        """Wait for batch `batch_no` of every rank; returns (counts per rank, frames in rank order or None).  If a rank had
        more records than the exchange capacity the frames are None even when asked for (counts are still exact): the
        caller gathers that batch some other way (dist.allgather_frames)."""
        counts = (c_uint32 * self._xchg_world)()
        n = c_uint32(0)
        out, ptr, cap = None, None, 0
        if want_frames:
            cap = self.max_frames * self._xchg_world
            out = np.zeros(cap, dtype=FRAME_DTYPE)
            ptr = out.ctypes.data_as(c_void_p)
        rc = self.lib.snrx_allgather(self.handle, batch_no, ptr, cap, counts, byref(n), timeout_ms)
        if rc == -6:                                           # SNRX_EOVERFLOW
            return list(counts), None
        self._check(rc)
        return list(counts), (out[: n.value].copy() if want_frames else None)

    # ------------------------------------------------------------------ SURVEY 8(f) N1: advertising analytics
    def adv_summary(self, want: bool = True) -> np.ndarray:
        """Per-record summaries (sender, PDU type, AD-structure fields: _abi.ADV_DTYPE) of the batch most recently
        returned by poll(), computed on the GPU from the HBM frame list; also folds the batch into the sender table.
        This is what Snout builds per btle_rx line (BtleMessage.fromraw -> BtlePDUPayload, message.py:205-237,
        advertising.py:113-307).  Call before the second-next process().  want=False only updates the table."""
        if not want:
            self._check(self.lib.snrx_ble_adv_summary(self.handle, None, 0, byref(c_uint32(0))))
            return np.zeros(0, dtype=_abi.ADV_DTYPE)
        return self._polled_list(self.lib.snrx_ble_adv_summary, _abi.ADV_DTYPE)

    def devices(self, reset: bool = False) -> np.ndarray:
        """The sender table (one _abi.DEVICE_DTYPE row per (AdvA, TxAdd), sorted by address) accumulated over every
        adv_summary() call: Snout's Device.get_unique bookkeeping (device.py:31-58) as packet counts, channel / PDU /
        AD masks, first and last position, latest company id."""
        n = c_uint32(0)
        self._check(self.lib.snrx_ble_devices(self.handle, None, 0, byref(n), 0))
        out = np.zeros(max(n.value, 1), dtype=_abi.DEVICE_DTYPE)
        self._check(self.lib.snrx_ble_devices(self.handle, out.ctypes.data_as(c_void_p), len(out), byref(n), 1 if reset else 0))
        out = out[: n.value]
        key = out["adv_a"].astype(np.uint64) @ (np.uint64(256) ** np.arange(6, dtype=np.uint64)) + (out["tx_add"].astype(np.uint64) << np.uint64(48))
        return out[np.argsort(key, kind="stable")]

    # ------------------------------------------------------------------ SURVEY 8(f) N3: BLE connections
    def connections(self) -> np.ndarray:
        """The CRC-ok CONNECT_REQs (_abi.CONN_DTYPE: AA, CRCInit, ChM, Hop, Interval, ...) among the records of the batch most
        recently returned by poll(): what btle_rx -o starts tracking (btle_rx.c:1476-1557, 2167-2282)."""
        return self._polled_list(self.lib.snrx_ble_connections, _abi.CONN_DTYPE)

    def follow(self, access_addr: int, crc_init: int) -> np.ndarray:
        """Search and decode the BLE channels of that batch again with a connection's access address and CRC init: the
        data-channel PDUs of the connection, from the slicer bit streams already in HBM (nothing is channelized twice)."""
        return self._polled_list(self.lib.snrx_ble_follow, FRAME_DTYPE, access_addr & 0xFFFFFFFF, crc_init & 0xFFFFFF)

    # ------------------------------------------------------------------ BLE 5 extended advertising
    def ble_aux(self) -> np.ndarray:
        """The auxiliary packets (AUX_ADV_IND, AUX_CHAIN_IND) that the ADV_EXT_INDs of the batch most recently returned by
        poll() point at, followed down their chains, on the 1M and 2M PHYs: one _abi.AUX_DTYPE entry per AuxPtr, found and
        decoded on the GPU from the batch's slicer bit streams (definition in include/snoutrx.h).  Wideband BLE modes; call
        before the second-next process()."""
        return self._polled_list(self.lib.snrx_ble_aux, _abi.AUX_DTYPE)

    # ------------------------------------------------------------------ BLE Long Range (LE Coded)
    def ble_coded(self) -> np.ndarray:
        """The ADV_EXT_INDs sent on the LE Coded PHY on channels 37..39 of the batch most recently returned by poll(),
        Viterbi-decoded, and the auxiliary packets they point at on every PHY, followed down their chains: one
        _abi.CODED_DTYPE entry per primary packet or AuxPtr, found and decoded on the GPU from the batch's slicer bit streams
        (definition in include/snoutrx.h).  Wideband BLE modes; call before the second-next process()."""
        return self._polled_list(self.lib.snrx_ble_coded, _abi.CODED_DTYPE)

    # ------------------------------------------------------------------ BLE periodic advertising
    def ble_periodic(self) -> np.ndarray:
        """The AUX_SYNC_IND trains that the SyncInfo fields of the batch's AUX_ADV_INDs (as ble_aux() finds them) describe, on
        the 1M and 2M PHYs: one _abi.SYNC_DTYPE entry per predicted event of a train inside the batch, with its counter,
        CSA#2 channel and window, found and decoded on the GPU from the batch's slicer bit streams (definition in
        include/snoutrx.h).  Wideband BLE modes; call before the second-next process()."""
        return self._polled_list(self.lib.snrx_ble_periodic, _abi.SYNC_DTYPE)

    # ------------------------------------------------------------------ BLE broadcast isochronous streams
    def ble_bis(self) -> np.ndarray:
        """The BIS subevents that the BIGInfo of the batch's AUX_SYNC_INDs (as ble_periodic() finds them) describes, on the
        1M and 2M PHYs: one _abi.BIS_DTYPE entry per subevent of a predicted BIG event inside the batch, with its BIS access
        address, CRC init, counter, channel, payload number and window, found and decoded on the GPU from the batch's slicer
        bit streams (definition in include/snoutrx.h).  Wideband BLE modes; call before the second-next process()."""
        return self._polled_list(self.lib.snrx_ble_bis, _abi.BIS_DTYPE)

    # ------------------------------------------------------------------ SURVEY 8(f) N2: Zigbee consumer path
    def zb_mac_summary(self) -> np.ndarray:
        """Per-record MAC summaries (_abi.ZBMAC_DTYPE: frame type, sequence number, PAN ids, addresses, inter-PAN / ZLL
        scan-response flags) of the batch most recently returned by poll(), computed on the GPU from the HBM frame list:
        what Snout reads off a scapy Dot15d4FCS tree per packet (zigbee.py:194-202, message.py:258-304)."""
        return self._polled_list(self.lib.snrx_zb_mac_summary, _abi.ZBMAC_DTYPE)

    # ------------------------------------------------------------------ per-frame radio metrics
    def frame_rf(self) -> np.ndarray:
        """Signal power, noise floor, SNR (dBFS / dB) and carrier offset (Hz) of every record of the batch most recently
        returned by poll(), aligned with it (_abi.RF_DTYPE; definition in include/snoutrx.h).  Needs rf_metrics=True;
        call before the second-next process()."""
        return self._polled_list(self.lib.snrx_frame_rf, _abi.RF_DTYPE)

    def frames_device(self) -> tuple[int, int]:
        f, c = c_void_p(), c_void_p()
        self._check(self.lib.snrx_frames_device(self.handle, byref(f), byref(c)))
        return f.value, c.value

    # ------------------------------------------------------------------ debug / parity
    def debug_stage(self, stage: int) -> np.ndarray:
        nb = c_uint64(0)
        self._check(self.lib.snrx_debug_stage(self.handle, stage, None, 0, byref(nb)))
        raw = np.zeros(nb.value, dtype=np.uint8)
        self._check(self.lib.snrx_debug_stage(self.handle, stage, raw.ctypes.data_as(c_void_p), nb.value, byref(nb)))
        caps, n_in = self._last
        n_out = n_in // self.decim
        if stage == _abi.STAGE_BLE_Q8:
            return raw.view(np.int8).reshape(caps, self.n_ble, n_out, 2)
        if stage == _abi.STAGE_CHAN_CF32:
            return raw.view(np.complex64).reshape(caps, self.n_zb if self.mode == MODE_ZB_WB16 else self.n_ble, n_out)
        if stage == _abi.STAGE_BLE_BITS:
            return raw.view(np.uint32).reshape(caps, self.n_ble, -1)
        if stage in (_abi.STAGE_ZB_DISC, _abi.STAGE_ZB_F):
            return raw.view(np.float32).reshape(caps, self.n_zb, -1)[:, :, :n_out]
        if stage == _abi.STAGE_ZB_NCHIPS:
            return raw.view(np.int64)
        if stage == _abi.STAGE_ZB_CHIPS:
            n_chains = len(self.debug_stage(_abi.STAGE_ZB_NCHIPS))
            return raw.view(np.float32).reshape(n_chains, -1)
        return raw
