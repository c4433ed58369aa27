/*
 * snoutrx.h -- C ABI of libsnoutrx.so, the B200-native IQ -> packet receive engine
 * that replaces Snout's two receive engines behind their own boundaries.
 *
 * Plain C: pointers and sizes only, no torch / C++ types.  Every entry point
 * returns 0 on success or a negative SNRX_E* code (snrx_strerror() explains it).
 * There is no CPU fallback anywhere behind this interface: if no CUDA device
 * is usable snrx_create() fails with SNRX_ENODEV.
 *
 * Which reference interface each entry point replaces (paths relative to the
 * nislab/snout tree):
 *
 *   snrx_create / snrx_destroy
 *       BLE   : process start of `btle_rx -c <ch> -g 6 -a 8e89bed6 -k 555555`
 *               (snout/util/btle.py:53-69; option table
 *               vendor/BTLE/host/btle-tools/src/btle_rx.c:1209-1294; board
 *               set-up config_run_board() btle_rx.c:623; crc_init_reorder()
 *               btle_rx.c:1801-1825 applied once at start, btle_rx.c:2335).
 *       Zigbee: construction of the flowgraph `top_block(channel=...)`
 *               (snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py:29-89).
 *   snrx_process
 *       BLE   : rx_callback() filling the ring (btle_rx.c:489-498) + the
 *               half-buffer loop calling receiver() (btle_rx.c:2341-2393,
 *               receiver() 2020-2155, search_unique_bits() 1369-1421,
 *               demod_byte() 1348-1367, scramble_byte() 1158-1163,
 *               crc_check() 1826-1848).
 *       Zigbee: the stream edges source -> quadrature_demod_cf -> (x - iir(x))
 *               -> clock_recovery_mm_ff -> packet_sink (top_block.py:52-73,
 *               80-89) and the sink's general_work()
 *               (scapy-radio/gnuradio/gr-zigbee/lib/packet_sink_scapy_impl.cc:158-374).
 *       Wideband modes additionally run the 96 Msps polyphase channelizer,
 *       which has no counterpart in the reference (it retunes one channel at
 *       a time: snout/util/btle.py:62, snout/core/radio.py:415).
 *   snrx_process_sc8
 *       the same with the reference's native sample format: int8 I,Q as delivered by
 *       hackrf_transfer.buffer to rx_callback() (btle_rx.c:489-498, IQ_TYPE btle_rx.c:204).
 *   snrx_poll
 *       BLE   : the printf()/fflush() of one line per frame (btle_rx.c:2137-2145,
 *               2383) that snout/core/pcontroller.py:115-131 reads back.
 *       Zigbee: message_port_pub() of the PSDU blob
 *               (packet_sink_scapy_impl.cc:333-349) -> UDP 127.0.0.1:52002
 *               (top_block.py:71) -> GnuradioSocket.recv
 *               (scapy-radio/scapy/scapy/modules/gnuradio.py:67-73).
 *   snrx_set_channel
 *       Zigbee: top_block.set_channel() via XMLRPC (top_block.py:94-96).
 *   snrx_debug_stage / snrx_debug_process_bits
 *       no reference counterpart: expose intermediate streams (quantised
 *       channel streams, discriminator output, soft chips) for parity tests,
 *       and run the BLE back end on given slicer bit streams.
 */
#ifndef SNOUTRX_H
#define SNOUTRX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNRX_ABI_VERSION 2

/* protocol ids = scapy-radio GnuradioPacket.proto values
 * (scapy-radio/scapy/scapy/layers/gnuradio.py:19-25) */
#define SNRX_PROTO_ZIGBEE 2
#define SNRX_PROTO_BLE    3

/* error codes */
#define SNRX_OK        0
#define SNRX_EINVAL   -1   /* bad argument / configuration            */
#define SNRX_ENODEV   -2   /* no usable CUDA device                   */
#define SNRX_ENOMEM   -3   /* host or device allocation failed        */
#define SNRX_ECUDA    -4   /* CUDA runtime error (see snrx_last_error) */
#define SNRX_ERANGE   -5   /* input larger than the configured capacity */
#define SNRX_EOVERFLOW -6  /* more candidates / frames than capacity  */
#define SNRX_ESTATE   -7   /* call out of sequence                    */

/* receive modes */
#define SNRX_MODE_BLE_NB     0  /* one BLE channel, 4 Msps cf32 in          (BASELINE config 1) */
#define SNRX_MODE_ZB_NB      1  /* one 802.15.4 channel, 4 Msps cf32 in     (config 2)          */
#define SNRX_MODE_ZB_WB16    2  /* 96 Msps in -> 16 Zigbee receivers        (config 3)          */
#define SNRX_MODE_BLE_WB40   3  /* 96 Msps in -> 40 BLE receivers           (config 4)          */
#define SNRX_MODE_MIXED_WB56 4  /* 96 Msps in -> 40 BLE + 16 Zigbee         (config 5)          */

/* geometry constants of the wideband channelizer (DESIGN.md "Channelizer") */
#define SNRX_WB_RATE      96000000
#define SNRX_WB_CENTER    2440000000ull
#define SNRX_WB_DECIM     24        /* 96 Msps -> 4 Msps per channel          */
#define SNRX_NB_RATE      4000000
#define SNRX_BLE_WINDOW   8192      /* btle_rx half buffer in IQ samples (btle_rx.c:180-182) */

/* One decoded frame.  Fixed 160 bytes so it can be all-gathered as-is. */
typedef struct snrx_frame {
    int64_t  sample_index;  /* channel-rate (4 Msps) IQ index, capture relative:
                               BLE: sample carrying access-address bit 0 (may be
                               -4..-1 at a window origin, btle_rx.c:1409);
                               Zigbee: input position of the chip completing the SFD */
    uint32_t capture_id;    /* index of the capture inside the processed batch */
    uint32_t window;        /* BLE: 8192-IQ window that reported it; Zigbee: segment */
    uint16_t channel;       /* BLE 0..39 / 802.15.4 11..26                    */
    uint8_t  proto;         /* SNRX_PROTO_*                                   */
    uint8_t  crc_ok;        /* BLE: CRC-24 matches (btle_rx prints CRC0); Zigbee: FCS-16 matches */
    uint8_t  lqi;           /* Zigbee: min(255,(sum/8)<<3) (packet_sink_scapy_impl.cc:334-335) */
    uint8_t  phase;         /* BLE: sample phase 0..3 of the hit                */
    uint16_t len;           /* valid bytes in bytes[]: BLE 2+payload+3, Zigbee PSDU length */
    uint32_t access_addr;   /* BLE                                            */
    uint8_t  bytes[132];    /* BLE: header|payload|crc (de-whitened); Zigbee: PSDU incl. FCS */
} snrx_frame_t;

/* Default Zigbee chain geometry: one clock-recovery + packet-sink chain per 4096 channel-rate samples
 * (1 ms), started 2048 samples early.  Part of the parity contract: the oracle runs the same segments.
 * (Measured on the oracle, tests/test_oracle_zigbee.py: how long the warm-up is does not change how close the
 * segmented receiver is to one unsegmented chain -- 2048 .. 131072 samples give the same frame agreement.) */
#define SNRX_ZB_SEGMENT_DEFAULT 4096
#define SNRX_ZB_PREHALO_DEFAULT 2048
/* Blocked DC tracker (a11): block length and memory in blocks; a time shard needs
 * (SNRX_ZB_IIR_MEMORY_BLOCKS + 1) * SNRX_ZB_IIR_BLOCK + zb_prehalo channel samples of pre halo. */
#define SNRX_ZB_IIR_BLOCK 2048
#define SNRX_ZB_IIR_MEMORY_BLOCKS 48
/* Span rule (also part of the contract): a CRC-failed 802.15.4 record whose sample_index lies inside the span of an
 * earlier CRC-ok record of the same (capture, channel) -- (2 + 2 * len) * 64 samples after its sample_index -- is not
 * reported: the reference's sequential packet sink is busy with that frame (packet_sink_scapy_impl.cc:247-359) and only
 * a chain restarted inside it can lock onto its payload chips.  Applied inside every batch; a caller that concatenates
 * time shards applies it once more across the shard boundary (snout_b200/stream.py zb_span_filter). */

typedef struct snrx_config {
    uint32_t abi_version;    /* must be SNRX_ABI_VERSION                                   */
    int32_t  device;         /* CUDA device ordinal                                        */
    int32_t  mode;           /* SNRX_MODE_*                                                */
    int32_t  channel;        /* NB modes: BLE 0..39 / Zigbee 11..26 ; ignored in WB modes  */
    uint32_t access_addr;    /* BLE `-a`  (default 0x8E89BED6, btle_rx.c:188)              */
    uint32_t crc_init;       /* BLE `-k`  as typed (0x555555, btle_rx.c:189)               */
    int32_t  zb_threshold;   /* packet sink threshold (10, top_block.py:67)                */
    float    quant_scale;    /* BLE: q = clamp(rint(x*quant_scale), -128, 127)             */
    uint64_t max_samples;    /* capacity: input samples per capture                        */
    uint32_t max_captures;   /* capacity: captures per snrx_process batch (wideband modes: <= 65535) */
    uint32_t max_frames;     /* capacity: frames per snrx_process batch                    */
    uint32_t zb_segment;     /* Zigbee: chain segment body, channel-rate samples (0 = SNRX_ZB_SEGMENT_DEFAULT) */
    uint32_t zb_prehalo;     /* Zigbee: chain warm-up, channel-rate samples (0 = SNRX_ZB_PREHALO_DEFAULT)   */
    uint32_t pfb_taps;       /* WB: prototype length, 384 or 768 (0 = default 384)         */
    uint32_t flags;          /* SNRX_F_*                                                   */
    uint32_t access_mask;    /* BLE `-m`: access-address bits that take part in the match
                                (0 = default 0xFFFFFFFF, btle_rx.c:1203,2301).  access_addr & mask must not be 0
                                (SNRX_EINVAL): such an address matches every run of zero decisions, so the
                                reference would decode a frame at every search origin, past the capture too */
    uint32_t reserved;       /* must be 0                                                  */
} snrx_config_t;

#define SNRX_F_KEEP_STREAMS 1u  /* also store channel streams so snrx_debug_stage can return them */
#define SNRX_F_RF_METRICS   2u  /* compute per-frame radio metrics in every batch (snrx_frame_rf) */

typedef struct snrx_stats {
    uint64_t samples_in;      /* input-rate samples consumed by the last snrx_process */
    uint64_t channel_samples; /* channel-rate samples produced (all channels)         */
    uint32_t candidates;      /* BLE access-address hits / Zigbee chains run          */
    uint32_t frames;          /* frames emitted                                       */
    uint32_t frames_crc_ok;
    uint32_t kernel_launches; /* kernels launched by the last snrx_process            */
    float    gpu_ms;          /* device time of the last snrx_process (CUDA events)   */
    float    gpu_ms_frontend; /* of which: channelizer / slicer kernel                */
} snrx_stats_t;

/* debug stages for snrx_debug_stage() */
#define SNRX_STAGE_BLE_Q8      1  /* int8 I,Q quantised channel streams [cap][ch][n][2]      */
#define SNRX_STAGE_BLE_BITS    2  /* uint32 slicer bit words [cap][ch][words], sample order  */
#define SNRX_STAGE_CHAN_CF32   3  /* cf32 channel streams [cap][ch][n] (WB modes)             */
#define SNRX_STAGE_ZB_DISC     4  /* f32 discriminator minus DC [cap][ch][stride] (stride = bytes/(4*cap*ch)) */
#define SNRX_STAGE_ZB_CHIPS    5  /* f32 soft chips [chain][chips_cap], chain = (cap, ch, segment)  */
#define SNRX_STAGE_ZB_F        6  /* f32 discriminator output before DC removal [cap][ch][stride] */
#define SNRX_STAGE_ZB_NCHIPS   7  /* int64 number of chips each chain produced [chain]            */

typedef struct snrx_handle snrx_t;

int  snrx_abi_version(void);
const char* snrx_strerror(int code);
const char* snrx_last_error(snrx_t* h);          /* detail text of the last failure (may be "") */

int  snrx_device_count(int* n);
int  snrx_create(snrx_t** h, const snrx_config_t* cfg);
void snrx_destroy(snrx_t* h);

/* Time shard of a longer capture (multi-GPU / streaming): the buffer handed to snrx_process
 * starts `pre_samples` before the shard body (read-only halo: channelizer history, Zigbee
 * warm-up) and may extend past it (post halo, so frames that start in the body can be
 * decoded completely).  Only frames anchored inside the body are reported, with the
 * sample_index / window they have in the whole capture, so the union over shards equals
 * the result of one call on the whole capture, bit for bit.  Requirements (channel rate):
 *   BLE    pre halo multiple of 128 (>= 128 unless the shard starts the capture), post halo
 *          >= 2048, body on the 8192-sample window grid;
 *          With SNRX_F_RF_METRICS and pfb_taps = 768 a wideband BLE shard that does not start the
 *          capture needs a pre halo >= 256: the noise window of a frame at the start of the body
 *          reaches 104 samples back and the channelizer needs 32 samples of history before it;
 *   Zigbee pre halo multiple of 2048 and >= 100352 + zb_prehalo unless the shard starts the
 *          capture (the DC tracker remembers 48 blocks of 2048 and the first block of a buffer
 *          starts without discriminator / channelizer history), post halo >= 16448, body on
 *          the zb_segment grid; zb_segment and zb_prehalo multiples of 2048, zb_segment a divisor
 *          or a multiple of 8192. */
typedef struct snrx_shard {
    uint64_t pre_samples;      /* input-rate samples of pre halo                                   */
    uint64_t body_samples;     /* input-rate samples of the body (0 = rest of the buffer)          */
    uint32_t first_window;     /* index inside the capture of the body's first 8192-sample window
                                  (channel rate); Zigbee segment = first_window * 8192 / zb_segment */
    uint32_t first_capture_id; /* capture_id reported for capture 0 of the batch                   */
} snrx_shard_t;

/* Run the receive path over a batch of `n_captures` captures, each `n_samples`
 * interleaved cf32 IQ samples long and `stride_samples` apart (input rate; 0 = n_samples).
 * `iq` is a host pointer (pageable or pinned; copied in chunks overlapped with
 * compute) or, if is_device_ptr != 0, a device pointer on cfg.device; 16-byte aligned.
 * `shard` is NULL for whole captures.  Asynchronous with respect to the host when
 * the input is a device pointer; results are collected with snrx_poll. */
int  snrx_process(snrx_t* h, const float* iq, uint32_t n_captures,
                  uint64_t n_samples, uint64_t stride_samples,
                  const snrx_shard_t* shard, int is_device_ptr);

/* snrx_process for captures stored as interleaved signed 8-bit I,Q -- the transfer format of the HackRF the
 * reference receives from (IQ_TYPE int8_t, btle_rx.c:204; rx_callback() copies exactly these bytes into the ring,
 * btle_rx.c:489-498).  Sample value x = q / 128 (exact), so with the narrow-band default quant_scale = 128 the
 * BLE path sees the reference's own int8 samples.  A quarter of the host->device bytes of cf32.  `iq` 16-byte
 * aligned, even stride for batches; sizes and strides count complex samples as in snrx_process. */
int  snrx_process_sc8(snrx_t* h, const int8_t* iq, uint32_t n_captures,
                      uint64_t n_samples, uint64_t stride_samples,
                      const snrx_shard_t* shard, int is_device_ptr);

/* Up to two batches may be queued (snrx_process, snrx_process, snrx_poll, ...): results are
 * collected oldest first.  snrx_poll waits for the oldest queued batch; *n_out = its number of
 * frames, in reference order (capture, channel, window, sample_index).  With out == NULL it only
 * reports the count; with out != NULL it copies up to `cap` frames and retires the batch.
 * snrx_poll_view retires the batch and returns a pointer to the engine's pinned host copy of the
 * frames (written by the kernels directly, no extra copy), valid until the second-next
 * snrx_process. */
int  snrx_poll(snrx_t* h, snrx_frame_t* out, uint32_t cap, uint32_t* n_out);
int  snrx_poll_view(snrx_t* h, const snrx_frame_t** frames, uint32_t* n_out);

/* Device-memory frame list / totals of the most recent snrx_process (valid once that batch has been
 * polled; the kernels write the list in HBM and k_export_frames copies it to the pinned host buffer). */
int  snrx_frames_device(snrx_t* h, void** frames_dev, void** count_dev);

/* Device-memory list of the frames of the batch most recently retired by snrx_poll / snrx_poll_view and
 * their count: the send buffer of the multi-GPU frame all-gather (SURVEY 8e; no host round trip, no copy).
 * The buffer holds max_frames records (those past the count are unspecified); the 160 bytes in front of it hold
 * {uint64 count, uint64 batch number (0, 1, ... per handle)}, so [header | records] can be sent as one block.  It stays
 * valid for two further snrx_process calls: it is overwritten by the third (each of the two lanes alternates between two lists). */
int  snrx_polled_frames_device(snrx_t* h, const snrx_frame_t** frames_dev, uint32_t* n_out);

/* ---- SURVEY 8(f) N1: advertising analytics on the decoded BLE records (what Snout does per btle_rx line:
 * BtleMessage.fromraw message.py:205-237 -> BtlePDUPayload advertising.py:113-307 -> Device device.py) ---- */
#define SNRX_ADV_FLAGS         0x0001  /* AD 0x01 present (ad_flags)                                   */
#define SNRX_ADV_UUID128       0x0002  /* AD 0x06                                                      */
#define SNRX_ADV_OOB           0x0004  /* AD 0x11 (oob_flags)                                          */
#define SNRX_ADV_SERVICE_DATA  0x0008  /* AD 0x16 (service_uuid)                                       */
#define SNRX_ADV_MANUFACTURER  0x0010  /* AD 0xff (company_id; Apple: apple_types / apple_action)      */
#define SNRX_ADV_UNKNOWN       0x0020  /* some other AD type (unknown_type = the last one)             */
#define SNRX_ADV_MALFORMED     0x0040  /* truncated where the reference parser raises / never returns  */
#define SNRX_ADV_SENDER        0x0080  /* adv_a holds the sender address                               */

/* snrx_adv_t.hints.  Low nibble: the first Nearby TLV (Apple type 0x10) of the record's Apple data -- 0 none, 1 present
 * without a version hint, 2 / 3 / 4 = the reference's 'iOS Version Hint' '10' / '11' / '12' (advertising.py:267-281). */
#define SNRX_HINT_NEARBY_MASK  0x0f
#define SNRX_HINT_FITBIT       0x10    /* the AD 0x06 field contains ba5689a6fabfa2bd01467d6e00fbabad (device.py:187-190)  */
/* snrx_device_t.model / .os codes */
#define SNRX_MODEL_NONE 0
#define SNRX_MODEL_FITBIT_CHARGE 1     /* 'Charge / Charge HR' (device.py:210-213)                             */
#define SNRX_MODEL_AIRPODS 2           /* Apple record of type 0x07 (device.py:214-219)                        */
#define SNRX_OS_NONE 0
#define SNRX_OS_UNDECIDED 1            /* a Nearby record without a version hint: the reference answers '-'    */
#define SNRX_OS_IOS10 2
#define SNRX_OS_IOS11 3
#define SNRX_OS_IOS12 4
#define SNRX_OS_WINDOWS10 5            /* company id 0x0006 (device.py:243-245)                                */
#define SNRX_VENDOR_NONE    0
#define SNRX_VENDOR_COMPANY 1          /* vendor_company holds the company id whose name Device.vendor returns */
#define SNRX_VENDOR_FITBIT  2          /* no company id in the first deciding packet, but the FitBit UUID: "FitBit" */

typedef struct snrx_adv {           /* one per record of the batch, 32 bytes */
    uint8_t  adv_a[6];      /* sender address as transmitted (btle_rx prints it reversed, btle_rx.c:1434-1441) */
    uint8_t  pdu_type;      /* header & 0x0f; 0xff: not a BLE record                                  */
    uint8_t  tx_add, rx_add;
    uint8_t  adv_len;       /* bytes of AD structures (PDU types 0, 2, 4, 6)                           */
    uint8_t  n_ad;          /* AD structures walked (AdvDataParser.get_ad_structure :74-91)            */
    uint8_t  ad_flags;      /* AD 0x01 value (last one wins, as in the reference's dict)               */
    uint16_t present;       /* SNRX_ADV_*                                                              */
    uint16_t company_id;    /* AD 0xff company (word16be() of the reference is little endian), 0xffff none */
    uint16_t service_uuid;  /* AD 0x16, 0xffff none                                                    */
    uint8_t  unknown_type;
    uint8_t  apple_action;  /* Apple Nearby (type 0x10) action code, 0xff none                         */
    uint8_t  oob_flags;     /* AD 0x11 value                                                           */
    uint8_t  hints;         /* SNRX_HINT_*: what Device.vendor / .model / .os look at (device.py:171-265)      */
    uint32_t apple_types;   /* bit t: Apple Continuity TLV type t (< 32) present (last Apple AD wins)   */
    uint32_t frame;         /* index of the record in the batch                                        */
} snrx_adv_t;

typedef struct snrx_device {        /* one per sender (AdvA, TxAdd), 64 bytes */
    uint8_t  adv_a[6];
    uint8_t  tx_add;
    uint8_t  ad_flags;      /* OR over its packets                                                     */
    uint32_t packets, crc_ok;
    uint64_t chan_mask;     /* bit c: seen on BLE channel c                                            */
    int64_t  first_index, last_index;     /* channel-rate position of its first / last packet (kept modulo 2^32 samples and
                                             2^16 captures inside the table: a stream longer than 17.9 minutes at 4 Msps
                                             should advance capture_id -- snrx_shard_t.first_capture_id -- per 2^32 samples) */
    uint32_t first_capture, last_capture; /* ... and their capture ids                                 */
    uint16_t pdu_mask;      /* bit t: PDU type t seen                                                  */
    uint16_t present;       /* OR of SNRX_ADV_* over its packets                                       */
    uint16_t company_id;    /* of its latest packet with manufacturer data, 0xffff none                */
    uint16_t vendor_company;/* Device.vendor (device.py:171-191): company id of its FIRST packet that carries one
                               (valid when vendor_kind == SNRX_VENDOR_COMPANY)                              */
    uint32_t apple_types;   /* OR over its packets                                                     */
    uint8_t  model;         /* Device.model (device.py:193-220): SNRX_MODEL_* decided by its first deciding packet */
    uint8_t  os;            /* Device.os (device.py:222-246): SNRX_OS_* decided by its first deciding packet   */
    uint8_t  vendor_kind;   /* SNRX_VENDOR_*                                                           */
    uint8_t  pad;
} snrx_device_t;

/* Summaries of the batch most recently retired by snrx_poll / snrx_poll_view (computed on the GPU from the device frame
 * list; call before the second-next snrx_process).  out may be NULL (only folds the batch into the device table).
 * *n_out = records of the batch (BLE and others; others have pdu_type 0xff). */
int  snrx_ble_adv_summary(snrx_t* h, snrx_adv_t* out, uint32_t cap, uint32_t* n_out);
/* The sender table accumulated by every snrx_ble_adv_summary call so far (unordered); reset != 0 clears it afterwards.
 * SNRX_EOVERFLOW if more than 2^18 distinct senders were seen (the extra ones were not recorded). */
int  snrx_ble_devices(snrx_t* h, snrx_device_t* out, uint32_t cap, uint32_t* n_out, int reset);

/* ---- SURVEY 8(f) N3: BLE connections.  btle_rx -o follows ONE connection by retuning its single channel on a wall-clock
 * schedule (receiver_controller, btle_rx.c:2167-2282: on a CRC-ok CONNECT_REQ it takes AA, CRCInit, ChM, Hop, Interval from
 * the fields parsed at btle_rx.c:1476-1557, hops hop_chan = (hop_chan + hop) % 37 and receives with the new access address
 * and crc_init_reorder(CRCInit)).  With all 40 channels channelized at once nothing has to be retuned or timed: the
 * CONNECT_REQs are picked out of the decoded records, and the data channels of the batch -- whose slicer bit streams are
 * still in HBM -- are searched and decoded AGAIN with the learned access address and CRC init. ---- */
typedef struct snrx_conn {          /* one per CRC-ok CONNECT_REQ (ADV PDU type 5, payload 34 bytes), 56 bytes */
    int64_t  sample_index;  /* of the CONNECT_REQ record                                                       */
    uint32_t capture_id;
    uint32_t frame;         /* index of the record in the batch                                                */
    uint32_t access_addr;   /* AA of the connection (payload bytes 12..15, little endian; btle_rx.c:1543-1546)  */
    uint32_t crc_init;      /* CRCInit as btle_rx.c:1505-1507 assembles it (byte 16 is the most significant):
                               the value to pass as crc_init (`-k`) for this connection                         */
    uint8_t  init_a[6], adv_a[6];   /* as transmitted (the reference stores them reversed for printing)          */
    uint16_t win_offset, interval, latency, timeout;
    uint8_t  chm[5];        /* channel map as transmitted (payload bytes 28..32)                               */
    uint8_t  win_size, hop, sca;
    uint8_t  channel;       /* advertising channel the request was heard on                                    */
    uint8_t  chm_full;      /* all 37 data channels used (the only maps btle_rx -o follows, btle_rx.c:2158-2163) */
    uint8_t  reserved[2];
} snrx_conn_t;

/* CONNECT_REQs (CRC ok) among the records of the batch most recently retired by snrx_poll / snrx_poll_view, in record order. */
int  snrx_ble_connections(snrx_t* h, snrx_conn_t* out, uint32_t cap, uint32_t* n_out);
/* Searches and decodes the BLE channels of that same batch again with another access address / CRC init (`-a` / `-k` of a
 * connection learned from snrx_ble_connections): *n_out frames in reference order, copied to out (up to cap).  The batch's
 * slicer bit streams are reused: nothing is channelized twice.  Call before the second-next snrx_process.  access_addr 0 is
 * refused (SNRX_EINVAL), like an all-zero compared address at snrx_create. */
int  snrx_ble_follow(snrx_t* h, uint32_t access_addr, uint32_t crc_init, snrx_frame_t* out, uint32_t cap, uint32_t* n_out);

/* ---- BLE 5 extended advertising: the auxiliary packets (AUX_ADV_IND, AUX_CHAIN_IND) that the ADV_EXT_INDs of a batch point
 * at, on the 1M and 2M PHYs, found and decoded from the batch's slicer bit streams (wideband BLE modes; nothing is
 * channelized twice).  No reference receiver exists for this: the definition below is the contract, and the GPU equals it
 * bit for bit on the engine's own bit streams (oracle/aux_oracle.py restates it).
 *
 * Pointer sources.  Depth 0: the records of the batch most recently retired by snrx_poll / snrx_poll_view with proto BLE,
 *   channel 37..39, crc_ok, access_addr 0x8E89BED6, PDU type 7 (header byte 0 & 0x0F), whose payload byte 0 gives an extended
 *   header length L >= 1 (bits 0..5) with 1 + L <= payload length, whose extended header flags (payload byte 1) have the AuxPtr
 *   bit (0x10) set, and whose extended header holds the fields in front of the AuxPtr (AdvA 6, TargetA 6, CTEInfo 1, ADI 2
 *   bytes, each if its flag bit 0..3 is set) and the AuxPtr itself: 2 + those fields + 3 <= 1 + L.
 *   Depth d > 0: the entries of depth d - 1 of this list with status OK, crc_ok, first == their own index, and the same
 *   AuxPtr conditions on their PDU (type 7 with an AuxPtr; the length is the full header byte 1).
 * AuxPtr (3 bytes a0 a1 a2): channel index a0 & 0x3F; CA (a0 >> 6) & 1; Offset Units (a0 >> 7): U = 30 or 300 us;
 *   Aux Offset A = a1 | (a2 & 0x1F) << 8; Aux PHY a2 >> 5 (SNRX_AUX_PHY_*).
 * Window.  s = the source's sample_index (AA bit 0, channel rate; for both PHYs AA bit 0 lies 32 samples after the first
 *   preamble sample).  O = A * U, ppm = 50 if CA else 500; the candidate positions n of the auxiliary packet's AA bit 0 are
 *     win_lo = s + floor(4 * O * (10^6 - ppm) / 10^6) - 8,   win_hi = s + ceil(4 * (O + U) * (10^6 + ppm) / 10^6) + 8
 *   (integer arithmetic, inclusive).
 * Search.  b[n] = the slicer decision of channel sample n of the aux channel (SNRX_STAGE_BLE_BITS); sps = 4 (1M) or 2 (2M).
 *   Decision n is usable when n + 1 < the buffer's channel samples (it pairs sample n with n + 1).  The earliest n in the
 *   window whose 32 decisions b[n + k sps] (k = 0..31) equal 0x8E89BED6 LSB first, all 32 bits compared.
 * Decode.  Byte j bit i = b[n + (32 + 8 j + i) sps]; the 2-byte header, len = header byte 1 (all 8 bits), then len + 3 more
 *   bytes; de-whitened with the x^7+x^4+1 LFSR seeded by the aux channel index (continued to 260 bytes); CRC-24 with
 *   crc_init 0x555555 (as snrx_create maps it) over 2 + len bytes, compared with the 3 bytes that follow.
 * Status (one per pointer, in this order of precedence):
 *   SNRX_AUX_DEPTH_LIMIT     depth > 15: not searched (chains are followed to depth 15)
 *   SNRX_AUX_BAD_CHANNEL     channel index > 36
 *   SNRX_AUX_UNSUPPORTED_PHY Coded or reserved PHY: not searched
 *   SNRX_AUX_OUTSIDE         win_lo or win_hi + 31 sps is not a usable decision of the buffer (the capture, or a shard's
 *                            pre-halo to post-halo span): not searched
 *   SNRX_AUX_NOT_FOUND       no match in the window
 *   SNRX_AUX_TRUNCATED       found, but the header's or the packet's last decision is not usable
 *   SNRX_AUX_OK              decoded; crc_ok says whether the CRC matches
 * Order and duplicates.  The list is ordered by depth, then by parent.  first = the list index of the earliest entry with
 *   status OK or TRUNCATED of the same (capture_id, channel, sample_index, phy), its own index if there is none; only
 *   entries with first == their own index start chains (the three ADV_EXT_INDs of an event normally point at one packet,
 *   and a chain that points back at itself ends there).
 * Shards.  Indices are whole-capture indices, as in the records.  A pointer whose window and packet lie inside both buffers
 *   gives the same entry in a time shard as in the whole capture; one that reaches past a shard's buffer is OUTSIDE there
 *   (pointers are not carried across shard boundaries). */
#define SNRX_AUX_OK              0
#define SNRX_AUX_NOT_FOUND       1
#define SNRX_AUX_OUTSIDE         2
#define SNRX_AUX_TRUNCATED       3
#define SNRX_AUX_UNSUPPORTED_PHY 4
#define SNRX_AUX_BAD_CHANNEL     5
#define SNRX_AUX_DEPTH_LIMIT     6
#define SNRX_AUX_PHY_1M    0
#define SNRX_AUX_PHY_2M    1
#define SNRX_AUX_PHY_CODED 2
#define SNRX_AUX_MAX_DEPTH 15
#define SNRX_AUX_MAX_BYTES 260    /* 2 header + 255 payload + 3 CRC */

typedef struct snrx_ble_aux {       /* one per pointer, 304 bytes */
    int64_t  sample_index;  /* AA bit 0 of the auxiliary packet (channel rate, capture relative); -1 unless OK / TRUNCATED */
    int64_t  win_lo, win_hi;/* the searched window of AA bit 0 positions, inclusive, capture relative                     */
    uint32_t capture_id;
    uint32_t parent;        /* depth 0: index of the ADV_EXT_IND record in the batch; deeper: index of the parent entry   */
    uint32_t first;         /* list index of the earliest entry that found the same packet (own index if none)           */
    uint8_t  depth;         /* 0 = pointed at by an ADV_EXT_IND, d = d links down a chain                                */
    uint8_t  channel;       /* AuxPtr channel index                                                                      */
    uint8_t  phy;           /* SNRX_AUX_PHY_*                                                                            */
    uint8_t  phase;         /* sample_index mod sps (0 unless OK / TRUNCATED)                                            */
    uint8_t  status;        /* SNRX_AUX_*                                                                                */
    uint8_t  crc_ok;        /* status OK and the CRC matches                                                             */
    uint16_t len;           /* valid bytes in bytes[]: 2 + header length + 3 (0 unless OK)                               */
    uint8_t  bytes[SNRX_AUX_MAX_BYTES];   /* de-whitened header | payload | CRC, zero past len                           */
} snrx_ble_aux_t;

/* The auxiliary packets of the batch most recently retired by snrx_poll / snrx_poll_view (definition above): *n_out entries,
 * copied to out (up to cap; out may be NULL to count).  Call before the second-next snrx_process.  SNRX_ESTATE without a
 * polled wideband BLE batch (SNRX_MODE_BLE_WB40 / SNRX_MODE_MIXED_WB56) or once its bit streams have been overwritten;
 * SNRX_ERANGE if cap is smaller than the list; SNRX_EOVERFLOW if the list would hold more than max_frames entries. */
int  snrx_ble_aux(snrx_t* h, snrx_ble_aux_t* out, uint32_t cap, uint32_t* n_out);

/* ---- BLE Long Range: the ADV_EXT_INDs sent on the LE Coded PHY on channels 37..39, found and Viterbi-decoded from the
 * batch's slicer bit streams, and the auxiliary packets they point at on every PHY (wideband BLE modes; nothing is
 * channelized twice).  No reference receiver exists for this: the definition below is the contract, and the GPU equals it
 * bit for bit on the engine's own bit streams (oracle/coded_oracle.py restates it).  Integer arithmetic only.
 *
 * Notation.  b[m] = the slicer decision of channel sample m (SNRX_STAGE_BLE_BITS); decision m is usable when m + 1 < the
 *   buffer's channel samples.  One LE Coded symbol is 4 channel samples (1 Msym/s, as LE 1M).
 * PHY (Core Vol 6 Part B 2.2, 3.3, as read here).  Encoder: rate 1/2, K = 4, state D1 | D2 << 1 | D3 << 2 with D1 the most
 *   recent input bit; a0 = u ^ D1 ^ D2 ^ D3 and a1 = u ^ D2 ^ D3 (G0 = 1+x+x^2+x^3, G1 = 1+x^2+x^3), a0 sent first.  Pattern
 *   mapper: S=8 maps 0 -> 0011 and 1 -> 1100, S=2 is the identity.  Packet: 80 preamble symbols (00111100 repeated); FEC
 *   block 1, always S=8, encoder from state 0: AA (32 bits) | CI (2 bits, LSB first) | TERM1 (3 zero bits); FEC block 2,
 *   encoder from state 0 again: whitened PDU | CRC-24 | TERM2 (3 zero bits), at S=8 if CI = 0 and at S=2 if CI = 1.
 *   Whitening and CRC (the channel's LFSR, init 0x555555) are applied before FEC.
 * Coded access address.  c[0..255] = 0x8E89BED6 encoded and mapped at S=8; P[j] = c[j >> 2], j = 0..1023.
 *   d(n) = the number of j in 0..1023 with b[n + j] != P[j], defined when n + 1023 is usable (otherwise infinite).
 * Primary packets.  On channels 37, 38 and 39 of every capture of the batch, n is a packet when d(n) <= T = 400 (noise: mean
 *   512, deviation 16), d(n) < d(m) for every m in [n - 16, n) and d(n) <= d(m) for every m in (n, n + 16] (a strict local
 *   minimum; the earliest wins ties).  sample_index = n (whole-capture index, as the records); a time shard reports the n
 *   inside its body only.  win_lo = win_hi = sample_index, parent = 0xFFFFFFFF, depth 0, phy SNRX_AUX_PHY_CODED.
 * Coding indicator.  Samples [n + 1024, n + 1184) carry CI and TERM1 (10 coded bits at 16 decisions).  ci = the v in 0..3
 *   whose coded (from the encoder state after the AA), mapped, sample-level pattern differs from b in the fewest places,
 *   the lower v on ties.  v = 2 or 3 is SNRX_AUX_RESERVED_CI: not decoded.
 * Viterbi.  Block 2 starts at n + 1184; coded bit k occupies the L = 16 (S=8) or L = 4 (S=2) decisions from n + 1184 + k L,
 *   and its branch metric is the number of them that differ from its sample-level pattern.  Add-compare-select keeps the
 *   predecessor with the smaller path metric, the one with D3 = 0 on ties; the start state has metric 0, the others 2^20.
 *   Header run: 40 info bits, traced back from the lowest-metric state at step 40 (lowest index on ties); its bits 0..15 are
 *   the whitened header and give len.  Full run: N = 8 len + 43 info bits, traced back from state 0 after TERM2.  The entry
 *   holds the full run's 2 + len + 3 de-whitened bytes, the CRC check, its final metric and d(n) (aa_errors).  If CI's, the
 *   header run's or the full run's last decision is not usable, the status is TRUNCATED.  The longest packet reaches
 *   n + 67 840.
 * Pointers.  Sources are the primary entries with status OK, crc_ok, first == own index and a PDU of type 7 with an AuxPtr
 *   (as for snrx_ble_aux), then, one depth down per round, the pointed entries meeting the same conditions.  The window is
 *   snrx_ble_aux's window shifted by the preamble lengths: s - P(source PHY) + P(target PHY) + [lo, hi], P = 32 for 1M and
 *   2M and 320 for Coded.  A 1M or 2M target is searched and decoded exactly as snrx_ble_aux does it.  A Coded target is
 *   OUTSIDE when win_lo or win_hi + 1023 is not a usable decision; else it takes the n of the window with the smallest
 *   d(n) <= T (earliest on ties; NOT_FOUND if none), decoded as above.  first, OUTSIDE, NOT_FOUND, BAD_CHANNEL and the
 *   depth limit follow snrx_ble_aux, with UNSUPPORTED_PHY for the reserved PHYs only and DEPTH_LIMIT beyond depth 16 (the
 *   same 15 chain links).
 * Order.  Primaries in (capture, channel, sample_index) order, then the pointer rounds by depth, then by parent.
 * Shards.  A packet whose decisions lie inside both buffers gives the same entry in a time shard as in the whole capture;
 *   one that reaches past a shard's buffer is TRUNCATED or OUTSIDE there (the default 2048-sample post-halo is shorter than
 *   most Coded packets: a shard needs a post-halo of 67 840 samples to decode every packet of its body). */
#define SNRX_AUX_RESERVED_CI     7
#define SNRX_CODED_T             400
#define SNRX_CODED_MAX_DEPTH     16

typedef struct snrx_ble_coded {     /* one per primary packet or pointer, 320 bytes */
    int64_t  sample_index;  /* start of the coded AA (Coded) or AA bit 0 (1M / 2M); -1 unless found                      */
    int64_t  win_lo, win_hi;/* the searched window, inclusive, capture relative (primaries: sample_index)                 */
    uint32_t capture_id;
    uint32_t parent;        /* list index of the pointing entry; 0xFFFFFFFF for primaries                                */
    uint32_t first;         /* list index of the earliest entry that found the same packet (own index if none)           */
    uint8_t  depth;         /* 0 = primary ADV_EXT_IND, d = d links from it                                              */
    uint8_t  channel;
    uint8_t  phy;           /* SNRX_AUX_PHY_*                                                                            */
    uint8_t  phase;         /* sample_index mod sps (4 for Coded)                                                        */
    uint8_t  status;        /* SNRX_AUX_*                                                                                */
    uint8_t  crc_ok;
    uint16_t len;           /* valid bytes in bytes[]: 2 + header length + 3 (0 unless OK)                               */
    uint8_t  ci;            /* coding indicator 0..3 of a Coded packet; 0xFF when not Coded or not reached               */
    uint8_t  reserved0;
    uint16_t aa_errors;     /* d(n) of a Coded packet                                                                    */
    uint32_t metric;        /* final path metric of the full Viterbi run (0 unless a Coded packet is OK)                 */
    uint8_t  bytes[SNRX_AUX_MAX_BYTES];   /* de-whitened header | payload | CRC, zero past len                           */
    uint8_t  reserved[8];
} snrx_ble_coded_t;

/* The Long Range packets of the batch most recently retired by snrx_poll / snrx_poll_view (definition above): *n_out
 * entries, copied to out (up to cap; out may be NULL to count).  State and capacity rules as snrx_ble_aux: SNRX_ESTATE
 * without a polled wideband BLE batch or once its bit streams have been overwritten; SNRX_ERANGE if cap is smaller than the
 * list; SNRX_EOVERFLOW if the list would hold more than max_frames entries. */
int  snrx_ble_coded(snrx_t* h, snrx_ble_coded_t* out, uint32_t cap, uint32_t* n_out);

/* ---- BLE periodic advertising: the AUX_SYNC_IND trains that the SyncInfo fields of a batch's AUX_ADV_INDs describe, on the
 * 1M and 2M PHYs, found and decoded from the batch's slicer bit streams (wideband BLE modes; nothing is channelized twice
 * and nothing hops).  No reference receiver exists for this: the definition below is the contract, and the GPU equals it
 * bit for bit on the engine's own bit streams (oracle/periodic_oracle.py restates it).  Integer arithmetic only.
 *
 * Train sources.  The entries of the list snrx_ble_aux returns for the same batch with status OK, crc_ok, first == their own
 *   index and a PDU of type 7 whose extended header (length L >= 1, 1 + L <= payload length) has the SyncInfo flag (0x20)
 *   set and holds the fields in front of it (AdvA 6, TargetA 6, CTEInfo 1, ADI 2, AuxPtr 3 bytes, each if flagged) and the
 *   18-byte SyncInfo: 2 + those fields + 18 <= 1 + L.  A SyncInfo with Sync Packet Offset 0, Interval < 6 or fewer than 2
 *   used channels is not a source.  One train per distinct (capture_id, access address): its source is the candidate with
 *   the smallest sample_index, the lower list index on ties.  Trains are ordered by their source's list index.
 * SyncInfo (18 bytes, little endian; Core Vol 6 Part B 2.3.4.6 as read here).  Bytes 0..1: Sync Packet Offset (13 bits) |
 *   Offset Units << 13 (U = 30 or 300 us) | Offset Adjust << 14 (adds 2 457 600 us).  Bytes 2..3: Interval (x 1.25 ms).
 *   Bytes 4..8: ChM (bits 0..36, bit c = data channel c used) | SCA << 37 (3 bits: ppm = 500, 250, 150, 100, 75, 50, 30,
 *   20).  Bytes 9..12: AA.  Bytes 13..15: CRCInit, reported and used as crc_init = c0 << 16 | c1 << 8 | c2 (c0..c2 in
 *   transmit order: snrx_conn_t.crc_init's and snrx_ble_follow's convention).  Bytes 16..17: paEventCounter.
 * Events.  Event k (any integer) has event_counter = (paEventCounter + k) mod 2^16, the source's PHY, and the channel of
 *   Channel Selection Algorithm #2 (Core Vol 6 Part B 4.5.8.3) for that counter: channelIdentifier = AA[31:16] ^ AA[15:0];
 *   prn_e = three rounds of PERM (bit reversal within each byte) then MAM (17 a + b mod 2^16, b = channelIdentifier) on
 *   counter ^ channelIdentifier, then ^ channelIdentifier; unmapped = prn_e mod 37; if unmapped is not used, the channel is
 *   used channel number (N prn_e) >> 16 in ascending order, N = the number of used channels.
 * Window.  s = the source's sample_index (AA bit 0 lies 32 samples after the first preamble sample on both PHYs), O = offset
 *   * U (+ 2 457 600 if Offset Adjust), I' = 1250 Interval us, p = the SCA's ppm, D_lo = O + k I', D_hi = O + U + k I':
 *     win_lo = s + early(D_lo) - 8,   win_hi = s + late(D_hi) + 8,
 *     early(D) = floor(4 D (10^6 - p) / 10^6) for D >= 0 and floor(4 D (10^6 + p) / 10^6) for D < 0,
 *     late(D)  = ceil(4 D (10^6 + p) / 10^6)  for D >= 0 and ceil(4 D (10^6 - p) / 10^6)  for D < 0
 *   (mathematical floor and ceiling, inclusive).  For k = 0 this is snrx_ble_aux's window with p from the SCA.
 * Listed events.  Every k with (a) win_hi - win_lo + 1 <= 2500 Interval (half the interval in samples) and (b)
 *   [win_lo, win_hi + 31 sps] meeting the buffer's usable decisions, in ascending k.  The width grows with |D| on both sides
 *   of D = 0 by 8 I' p / 10^6 >= 1.2 samples per event, more than the two roundings can take back, so both rules and the
 *   list hold one contiguous range of k.  Rule (a) keeps a train's windows (with the 31 sps span) disjoint, and two trains
 *   never share an AA, so no packet is listed twice.
 * Search, decode and status.  As snrx_ble_aux, with the train's AA (all 32 bits compared) and crc_init, the earliest match in
 *   the window, len = header byte 1 (all 8 bits), de-whitened by the event's channel:
 *   SNRX_AUX_OUTSIDE (win_lo or win_hi + 31 sps is not a usable decision: not searched), SNRX_AUX_NOT_FOUND,
 *   SNRX_AUX_TRUNCATED (the header's or the packet's last decision is not usable), SNRX_AUX_OK (crc_ok says whether the CRC
 *   matches).
 * Order.  Trains in source order, each train's events in ascending k.
 * Shards.  Indices are whole-capture indices.  Each shard predicts from its own sources; trains are not carried across
 *   shards, and an event whose window leaves a shard's buffer is OUTSIDE there or not listed.
 * Not covered: AUX_CHAIN_INDs an AUX_SYNC_IND points at (its bytes are kept), trains on LE Coded, periodic advertising with
 *   responses, BIG / BIS data, and re-anchoring on found events (windows are predicted from the source alone). */
#define SNRX_SYNC_MIN_INTERVAL 6

typedef struct snrx_ble_sync {      /* one per listed event of a train, 320 bytes */
    int64_t  sample_index;  /* AA bit 0 of the AUX_SYNC_IND (channel rate, capture relative); -1 unless OK / TRUNCATED       */
    int64_t  win_lo, win_hi;/* the searched window of AA bit 0 positions, inclusive, capture relative                     */
    uint32_t capture_id;
    uint32_t source;        /* index in the snrx_ble_aux list of the AUX_ADV_IND whose SyncInfo the train comes from      */
    uint32_t access_addr;   /* the train's AA                                                                            */
    uint32_t crc_init;      /* the train's CRCInit as c0 << 16 | c1 << 8 | c2 (the value snrx_ble_follow takes)            */
    int32_t  event;         /* k: events after (negative: before) the one the SyncInfo points at                         */
    uint16_t event_counter; /* (paEventCounter + k) mod 2^16                                                              */
    uint16_t interval;      /* in 1.25 ms units                                                                          */
    uint8_t  channel;       /* CSA#2 channel of the event                                                                */
    uint8_t  phy;           /* SNRX_AUX_PHY_1M or SNRX_AUX_PHY_2M (the source's)                                        */
    uint8_t  phase;         /* sample_index mod sps (0 unless OK / TRUNCATED)                                            */
    uint8_t  status;        /* SNRX_AUX_OK, _NOT_FOUND, _OUTSIDE or _TRUNCATED                                           */
    uint8_t  crc_ok;        /* status OK and the CRC matches                                                             */
    uint8_t  sca;           /* SyncInfo SCA 0..7                                                                         */
    uint16_t len;           /* valid bytes in bytes[]: 2 + header length + 3 (0 unless OK)                               */
    uint8_t  bytes[SNRX_AUX_MAX_BYTES];   /* de-whitened header | payload | CRC, zero past len                           */
    uint8_t  reserved[4];
} snrx_ble_sync_t;

/* The periodic-advertising events of the batch most recently retired by snrx_poll / snrx_poll_view (definition above):
 * *n_out entries, copied to out (up to cap; out may be NULL to count).  Builds the snrx_ble_aux list itself first.  State
 * and capacity rules as snrx_ble_aux: SNRX_ESTATE without a polled wideband BLE batch or once its bit streams have been
 * overwritten; SNRX_ERANGE if cap is smaller than the list; SNRX_EOVERFLOW if the aux list or this list would hold more than
 * max_frames entries. */
int  snrx_ble_periodic(snrx_t* h, snrx_ble_sync_t* out, uint32_t cap, uint32_t* n_out);

/* ---- BLE broadcast isochronous streams: the BIS subevents that the BIGInfo in a batch's AUX_SYNC_INDs describes, on the 1M
 * and 2M PHYs, found and decoded from the batch's slicer bit streams (wideband BLE modes; nothing is channelized twice and
 * nothing hops).  No reference receiver exists for this: the definition below is the contract, and the GPU equals it bit for
 * bit on the engine's own bit streams (oracle/bis_oracle.py restates it).  Integer arithmetic only.
 *
 * Carriers.  The entries of the list snrx_ble_periodic returns for the same batch with status OK, crc_ok and a PDU of type 7
 *   whose extended header has length L >= 1 with 1 + L <= payload length and holds its flagged fields (AdvA 6, TargetA 6,
 *   CTEInfo 1, ADI 2, AuxPtr 3, SyncInfo 18, TxPower 1 bytes); the header bytes past them are the ACAD.  The ACAD is walked
 *   as AD structures (length | type | value), stopping at a length-0 structure or one that overruns it; its first structure
 *   of type 0x2C must have length byte 34 (an unencrypted BIGInfo, 33 bytes) or 58 (encrypted, 57 bytes), and that BIGInfo
 *   must be valid (below).
 * BIGInfo (little endian; Core Vol 6 Part B 2.3.4.8 as read here).  Bytes 0..3: BIG_Offset (14 bits) | BIG_Offset_Units << 14
 *   (U = 30 or 300 us) | ISO_Interval << 15 (12 bits, x 1.25 ms) | Num_BIS << 27 (5).  Bytes 4..7: NSE (5) | BN << 5 (3) |
 *   Sub_Interval << 8 (20, us) | PTO << 28 (4).  Bytes 8..11: BIS_Spacing (20, us) | IRC << 20 (4) | Max_PDU << 24 (8).
 *   Byte 12: RFU.  Bytes 13..16: SeedAccessAddress (SAA).  Bytes 17..20: SDU_Interval (20) | Max_SDU << 20 (12).  Bytes
 *   21..22: BaseCRCInit.  Bytes 23..27: ChM (bits 0..36) | PHY << 37 (3: 0 = 1M, 1 = 2M, 2 = Coded).  Bytes 28..32:
 *   bisPayloadCount (39 bits) | Framing << 39.  Bytes 33..56 (encrypted only): GIV (8) and GSKD (16).
 *   Valid: Num_BIS, BN, NSE >= 1, NSE mod BN = 0, 1 <= IRC <= NSE / BN; ISO_Interval >= 4; PHY 1M or 2M; at least 2 used
 *   channels; (Num_BIS - 1) BIS_Spacing + (NSE - 1) Sub_Interval < 1250 ISO_Interval; S_min > 0, where S_min (the spacing of
 *   two packets of one BIS, us) = min(Sub_Interval, 1250 ISO_Interval - (NSE - 1) Sub_Interval), or 1250 ISO_Interval when
 *   NSE = 1.
 * BIGs.  One per distinct (capture_id, SAA): its source is the carrier with the smallest sample_index, the lower list index
 *   on ties; BIGs are ordered by their source's index in the periodic list.  Everything is predicted from the source alone.
 * BIS n = 1..Num_BIS (Vol 6 Part B 2.1.2 as read here).  AA_n = SAA ^ DW_n with D = (35 n + 42) mod 128 (bits D6..D0) and
 *   the diversifier word DW_n, from bit 31 down to bit 0: D0 D0 D0 D0 D0 D0 D1 D6 | D1 0 D5 D4 0 D3 D2 0 | 16 zero bits.
 *   The 24-bit CRCInit is BaseCRCInit << 8 | n, sent least significant byte first, so crc_init (c0 << 16 | c1 << 8 | c2 in
 *   transmit order: snrx_conn_t.crc_init's and snrx_ble_follow's convention) = n << 16 | (BaseCRCInit & 0xFF) << 8 |
 *   BaseCRCInit >> 8.  A BIS whose AA_n is 0 is not searched (its entries are NOT_FOUND): an all-zero address would match
 *   any run of 32 zero decisions.
 * Events.  Event k (any integer) has event_counter E_k = (floor(bisPayloadCount / BN) + k) mod 2^16.  Its subevent (n, se),
 *   se = 0..NSE-1, has D_lo = O + 1250 k ISO_Interval + (n - 1) BIS_Spacing + se Sub_Interval (us), O = BIG_Offset U,
 *   D_hi = D_lo + U, measured from s = the source's sample_index (AA bit 0 lies 32 samples after the first preamble sample on
 *   both PHYs), and p = the ppm of the source's train's SCA (the BIGInfo carries no SCA; this is the reading used here):
 *     win_lo = s + early(D_lo) - 8,   win_hi = s + late(D_hi) + 8   (early / late as snrx_ble_sync_t's windows).
 * Channel (Vol 6 Part B 4.5.8.3 as read here).  Subevent 0: CSA#2 of E_k with AA_n and ChM (as snrx_ble_sync_t's events).
 *   Subevents se >= 1: prnSubEvent_lu starts at the event's prn_s (prn_e before its final ^ channelIdentifier); each
 *   subevent sets prnSubEvent_lu = MAM(PERM(prnSubEvent_lu)), prnSubEvent_se = prnSubEvent_lu ^ channelIdentifier, and takes
 *   used channel number index = (lastIndex + d + ((prnSubEvent_se (N - 2 d + 1)) >> 16)) mod N in ascending order, with
 *   d = max(1, max(min(3, N - 5), min(11, (N - 10) / 2))), N = the number of used channels and lastIndex the used-channel
 *   number of the previous subevent (of subevent 0 to start).
 * Payload number (Vol 6 Part B 4.4.6.6 as read here).  g = se / BN, i = se mod BN:
 *   payload_number = ((floor(bisPayloadCount / BN) + k + (g < IRC ? 0 : PTO (g - IRC + 1))) mod 2^39) BN + i.
 * Listed events.  k_c = the first k with D_lo(1, 0) >= 0.  Event k is listed when (a) every subevent window of every event
 *   from k to k_c (inclusive) is at most 2 S_min samples long, and (b) [win_lo(1, 0), win_hi(Num_BIS, NSE - 1) + 31 sps]
 *   meets the buffer's usable decisions.  A listed event contributes all its Num_BIS x NSE entries; an entry whose own
 *   [win_lo, win_hi + 31 sps] leaves the usable decisions is OUTSIDE.  Two packets of one BIS are at least S_min us =
 *   4 S_min samples apart, so a window of at most 2 S_min samples (with the 31 sps address span) ends before the next one
 *   of its BIS starts: no packet is listed twice.
 * Search, decode and status.  As snrx_ble_sync_t's, with AA_n (all 32 bits), crc_init_n and the subevent's channel, at 4
 *   samples per symbol on 1M and 2 on 2M (the BIGInfo's PHY): OUTSIDE, NOT_FOUND, TRUNCATED or OK with crc_ok.  The payload
 *   of an encrypted BIS is reported as sent (its MIC is part of len).
 * Order.  BIGs in source order; within a BIG ascending k, then BIS number, then subevent.
 * Shards.  Indices are whole-capture indices.  Each shard predicts from its own carriers; BIGs are not carried across shards.
 * Spec-dependent pieces, unverified here against the specification's sample data: the BIGInfo bit layout, the diversifier
 *   word, the subevent channel mapping and the payload numbering (DESIGN.md section 4).
 * Not covered: decrypting encrypted BISes (needs the Broadcast_Code), BIG Control subevents (after a channel map update the
 *   entries are NOT_FOUND), BIGs on LE Coded, re-anchoring on found events, ISOAL SDU reassembly, connected isochronous
 *   streams. */
#define SNRX_BIS_ENCRYPTED 0x01     /* snrx_ble_bis_t.flags */
#define SNRX_BIS_FRAMED    0x02

typedef struct snrx_ble_bis_entry { /* one per subevent of a listed BIG event, 336 bytes */
    int64_t  sample_index;  /* AA bit 0 of the BIS PDU (channel rate, capture relative); -1 unless OK / TRUNCATED            */
    int64_t  win_lo, win_hi;/* the searched window of AA bit 0 positions, inclusive, capture relative                     */
    uint64_t payload_number;/* the payload this subevent carries (definition above)                                      */
    uint32_t capture_id;
    uint32_t source;        /* index in the snrx_ble_periodic list of the AUX_SYNC_IND whose BIGInfo the BIG comes from   */
    uint32_t access_addr;   /* AA_n                                                                                      */
    uint32_t crc_init;      /* crc_init_n as c0 << 16 | c1 << 8 | c2 (the value snrx_ble_follow takes)                     */
    int32_t  event;         /* k: BIG events after (negative: before) the one the BIGInfo points at                      */
    uint16_t event_counter; /* E_k                                                                                         */
    uint8_t  bis;           /* n, 1..Num_BIS                                                                              */
    uint8_t  subevent;      /* se, 0..NSE-1                                                                               */
    uint8_t  channel;       /* the subevent's data channel                                                               */
    uint8_t  phy;           /* SNRX_AUX_PHY_1M or SNRX_AUX_PHY_2M (the BIGInfo's)                                       */
    uint8_t  phase;         /* sample_index mod sps (0 unless OK / TRUNCATED)                                            */
    uint8_t  status;        /* SNRX_AUX_OK, _NOT_FOUND, _OUTSIDE or _TRUNCATED                                           */
    uint8_t  crc_ok;        /* status OK and the CRC matches                                                             */
    uint8_t  flags;         /* SNRX_BIS_ENCRYPTED (a 57-byte BIGInfo) | SNRX_BIS_FRAMED                                   */
    uint16_t len;           /* valid bytes in bytes[]: 2 + length byte + 3 (0 unless OK)                                 */
    uint8_t  bytes[SNRX_AUX_MAX_BYTES];   /* de-whitened header | payload | CRC, zero past len                           */
    uint8_t  reserved[12];
} snrx_ble_bis_t;

/* The BIS subevents of the batch most recently retired by snrx_poll / snrx_poll_view (definition above): *n_out entries,
 * copied to out (up to cap; out may be NULL to count).  Builds the snrx_ble_aux and snrx_ble_periodic lists itself first.
 * State and capacity rules as snrx_ble_periodic: SNRX_ESTATE without a polled wideband BLE batch or once its bit streams
 * have been overwritten; SNRX_ERANGE if cap is smaller than the list; SNRX_EOVERFLOW if the aux list, the periodic list or
 * this list would hold more than max_frames entries. */
int  snrx_ble_bis(snrx_t* h, snrx_ble_bis_t* out, uint32_t cap, uint32_t* n_out);

/* ---- SURVEY 8(f) N2: the Zigbee consumer path on the decoded 802.15.4 records (what Snout does per datagram:
 * RFtap(pkt) -> Dot15d4FCS dissection, snout/util/zigbee.py:194-202; ZigbeeMessage.fromraw, snout/core/message.py:258-304;
 * the touchlink scan's haslayer(ZLLScanResponse), zigbee.py:176-192) ---- */
#define SNRX_ZBMAC_SECURITY           0x0001  /* FCF security enabled                                        */
#define SNRX_ZBMAC_PENDING            0x0002  /* FCF frame pending                                           */
#define SNRX_ZBMAC_ACKREQ             0x0004  /* FCF acknowledgement request                                 */
#define SNRX_ZBMAC_PANID_COMPRESS     0x0008  /* FCF PAN id compression                                      */
#define SNRX_ZBMAC_DEST_PANID         0x0010  /* dest_panid holds a value                                    */
#define SNRX_ZBMAC_DEST_ADDR          0x0020  /* dest_addr holds a value (dest_mode 2: 16 bit, 3: 64 bit)    */
#define SNRX_ZBMAC_SRC_PANID          0x0040
#define SNRX_ZBMAC_SRC_ADDR           0x0080
#define SNRX_ZBMAC_INTERPAN           0x0100  /* data frame whose payload is a ZigBee inter-PAN stub NWK frame */
#define SNRX_ZBMAC_ZLL                0x0200  /* ... carrying a ZLL commissioning cluster command (zll_command) */
#define SNRX_ZBMAC_ZLL_SCAN_RESPONSE  0x0400  /* ... which is a scan response (what the touchlink scan collects) */
#define SNRX_ZBMAC_NO_ADDRESSING      0x0800  /* an address mode without a length (none / reserved): the reference dissector
                                                 raises (dot15d4.py:60-63) and yields no addressing fields               */
#define SNRX_ZBMAC_MALFORMED          0x4000  /* the record ends inside a field the header announces          */
#define SNRX_ZBMAC_NOT_ZIGBEE         0x8000  /* the record is not an 802.15.4 record                         */

typedef struct snrx_zbmac {         /* one per record of the batch, 40 bytes */
    uint64_t dest_addr, src_addr;   /* short addresses in the low 16 bits                                      */
    uint16_t dest_panid, src_panid;
    uint16_t fcf;                   /* frame control field as transmitted (little endian)                      */
    uint16_t present;               /* SNRX_ZBMAC_*                                                            */
    uint8_t  seqnum;
    uint8_t  frame_type;            /* 0 beacon, 1 data, 2 ack, 3 command (0xff: record too short)             */
    uint8_t  dest_mode, src_mode;   /* addressing modes 0 none, 2 short, 3 long                                */
    uint8_t  cmd_id;                /* MAC command id (command frames), else 0xff                              */
    uint8_t  payload_off;           /* offset of the MAC payload inside the PSDU                               */
    uint8_t  zll_command;           /* ZLL commissioning command id, 0xff none                                 */
    uint8_t  reserved;
    uint16_t cluster, profile;      /* inter-PAN APS stub cluster / profile                                    */
    uint32_t frame;                 /* index of the record in the batch                                        */
} snrx_zbmac_t;

/* Summaries of the batch most recently retired by snrx_poll / snrx_poll_view, computed on the GPU from the device frame
 * list (call before the second-next snrx_process).  *n_out = records of the batch (BLE records get SNRX_ZBMAC_NOT_ZIGBEE). */
int  snrx_zb_mac_summary(snrx_t* h, snrx_zbmac_t* out, uint32_t cap, uint32_t* n_out);

/* ---- Radio metrics of every decoded frame (engine created with SNRX_F_RF_METRICS): signal power, noise floor, SNR and
 * carrier offset, what packet sniffers report beside each packet (the PHDR fields of LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR,
 * the RFtap power / noise / snr / freqofs fields).  Computed inside the batch, from the input, by k_frame_rf.
 *
 * Definition.  s = the record's sample_index (channel rate, capture relative); y[m] = the frame's channel samples:
 *   wideband modes    the channelizer's own definition (DESIGN.md "Channelizer") for the bin of the frame's channel
 *                     (snrx_ble_channel_bin / snrx_zigbee_channel_bin) with the prototype of its protocol
 *                     (snrx_pfb_prototype(mode, pfb_taps)); x = 0 outside the buffer;
 *   narrow-band modes y = the input itself (sc8 input: q / 128, the value the engine expands it to).
 * Windows, half-open [a, b) relative to s:
 *   BLE       signal / CFO [s-24, s+120)   preamble bits 2..7 and access-address bits 0..29
 *             noise        [s-104, s-40)   64 samples ending 8 before the preamble
 *   802.15.4  signal / CFO [s-392, s-136)  4 whole preamble symbol periods ending 8 before the nominal SFD start s-128
 *             noise        [s-720, s-656)  64 samples ending 16 before the nominal SHR start s-640
 *   (Measured on synthetic bursts of known start, narrow band and through the synthesis filterbank at both prototype
 *   lengths: the BLE sample_index lies 1 (narrow band) or 0.5 (wideband, after the filter delays) samples before the
 *   nominal position of AA bit 0, the 802.15.4 one 3..5 samples before the nominal PHR start -- inside the guards, so the
 *   windows stay where the nominal positions put them.)
 *   power_dbfs = 10 log10(mean |y[m]|^2) over the signal window, noise_dbfs the same over the noise window (0 dBFS = |x| = 1
 *   at the input; the prototypes have unity DC gain); a mean below 1e-20 reads -200.  snr_db = power_dbfs - noise_dbfs.
 *   cfo_hz = fs / 2 pi * wrap(arg(sum_{m=a}^{b-1} y[m] conj(y[m-1])) - theta0), fs = 4e6, over the signal window (so it also
 *   reads y[a-1]); theta0 = arg sum_m exp(j dtheta_ref[m]) over the same m, dtheta_ref = the per-sample phase increment of the
 *   zero-offset reference waveform:
 *     BLE       the GFSK waveform (h = 0.5, 4 samples per bit, the 16 Gaussian taps of BT 0.5 -- snrx_tx_burst_t, synth.py)
 *               of the 40 known bits -- preamble (0xAA, or 0x55 when AA bit 0 is 1) then the record's access_addr, LSB first --
 *               with the burst's first sample at s - 39 (the measured position above); computed per frame;
 *     802.15.4  the preamble is periodic in 64 samples, so theta0 over whole periods is one constant: SNRX_RF_ZB_THETA0.
 *   Positive cfo_hz = carrier above the channel centre (the sign of snrx_tx_burst_t.cfo_hz).
 *   A window that reaches before channel sample 0 of the capture, or of the buffer, or past the buffer's end is not
 *   evaluated: its values are NaN and its valid bits are clear (snr_db is NaN unless both windows are valid). */
#define SNRX_RF_POWER 0x01     /* power_dbfs valid (the signal window lies inside the buffer)  */
#define SNRX_RF_NOISE 0x02     /* noise_dbfs valid                                             */
#define SNRX_RF_CFO   0x04     /* cfo_hz valid (same window as the power)                      */
#define SNRX_RF_ZB_THETA0 0.12435499454676144   /* atan(1/8): 36 of every 64 preamble increments are +pi/4, 28 are -pi/4 */

typedef struct snrx_frame_rf {      /* one per record of the batch, 40 bytes */
    int64_t  sample_index;  /* key fields copied from the record, so that consumers can join after reordering / filtering */
    uint32_t capture_id;
    uint32_t frame;         /* index of the record in the batch                                                */
    uint16_t channel;
    uint8_t  proto;
    uint8_t  valid;         /* SNRX_RF_*                                                                       */
    float    power_dbfs, noise_dbfs, snr_db, cfo_hz;
    uint32_t reserved;
} snrx_frame_rf_t;

/* Radio metrics of the records of the batch most recently retired by snrx_poll / snrx_poll_view, in record order
 * (*n_out = records of the batch; out may be NULL; SNRX_ERANGE if cap is smaller than the batch).  Call before the
 * second-next snrx_process.  SNRX_ESTATE if the engine was created without SNRX_F_RF_METRICS or nothing has been polled. */
int  snrx_frame_rf(snrx_t* h, snrx_frame_rf_t* out, uint32_t cap, uint32_t* n_out);

/* ---- SURVEY 8(e) / a19: the one exchange of the path -- every engine of a node gets every engine's frame records.
 * No reference counterpart (the reference runs on one host CPU); north_star: "NCCL over NVLink is used only to allgather
 * the decoded-frame records".  Here the gather needs no collective kernel at all: once the engines are connected, the
 * kernel that exports a batch's frame list (k_export_frames) also stores the records -- only the 16-byte pieces a record
 * uses -- and then a {count, batch} header straight into a receive slot in every peer's HBM over NVLink / NVSwitch
 * (peer pointers obtained through CUDA IPC).  Nothing is launched or waited for per batch on the host, and no SM-resident
 * collective waits for the slowest rank beside the channelizer.
 *
 *   snrx_exchange_create   allocates this engine's receive area (8 slots x world x (1 + cap_records) records) and returns
 *                          its 64-byte CUDA IPC handle; the caller passes the handles around (MPI, torch.distributed,
 *                          a file: 64 bytes per rank) ...
 *   snrx_exchange_connect  ... and hands all of them in, in rank order; every later batch is pushed to every rank.
 *   snrx_allgather         waits until batch `batch_no` (0, 1, ... = the order of snrx_process calls on every engine) of
 *                          all ranks has arrived here; counts[r] = records of rank r; with out != NULL the records are
 *                          copied out in rank order (*n_out = their number).  Collective discipline: every rank calls it
 *                          for every batch, in order, and before it queues batch_no + 4 (a slot is reused after 8 batches).
 *                          SNRX_EOVERFLOW if some rank had more than cap_records records in that batch (the caller falls back
 *                          to its own two-phase gather for that batch), SNRX_ESTATE after timeout_ms without the batch. */
#define SNRX_XCHG_HANDLE_BYTES 64
#define SNRX_XCHG_SLOTS 8
#define SNRX_XCHG_MAX_WORLD 16
int  snrx_exchange_create(snrx_t* h, uint32_t rank, uint32_t world, uint32_t cap_records, void* handle_out);
int  snrx_exchange_connect(snrx_t* h, const void* handles);
int  snrx_allgather(snrx_t* h, uint64_t batch_no, snrx_frame_t* out, uint32_t cap, uint32_t* counts, uint32_t* n_out,
                    uint32_t timeout_ms);

/* ---- SURVEY 8(f) N4: the transmit side on the GPU -- synthetic / replay captures generated where they are consumed.
 * Waveforms as the reference's transmitters state them: GFSK per vendor/BTLE/host/btle-tools/src/btle_tx.c:1111-1149
 * (gen_sample_from_phy_bit, float version; h = 0.5, 4 samples per symbol, 16 Gaussian taps :103-128), half-sine O-QPSK per
 * snout/grc-blocks/transmitter_OQPSK.py:96-111 with the SHR / PHR of gr-zigbee preamble_prefixer_scapy_impl.cc:48-52,67-88.
 * Every burst is one frame: the caller provides its bits / bytes and where it goes (the schedule is a few bytes per frame
 * and is drawn on the host, snout_b200/synth.py); the GPU modulates, places the bursts in their 4 Msps channel streams,
 * lifts the streams to 96 Msps through a 96-bin synthesis filterbank (x24 polyphase interpolation, 384 taps, and the
 * rotation to the bin centre) and adds white Gaussian noise from a counter-based generator (a function of seed and
 * sample index only: the same call gives the same capture). */
typedef struct snrx_tx_burst {
    int64_t  start;        /* channel-rate (4 Msps) sample index of the burst's first sample                              */
    uint32_t data_offset;  /* offset of the burst's data in `data`                                                       */
    uint32_t n_units;      /* BLE: PHY bits (preamble | access address | whitened PDU + CRC, LSB first, 8 per data byte);
                              802.15.4: PPDU bytes (SHR | PHR | PSDU)                                                     */
    uint16_t bin_slot;     /* index into `bins`: the filterbank bin (snrx_*_channel_bin) the burst is sent on             */
    uint8_t  proto;        /* SNRX_PROTO_BLE (GFSK) or SNRX_PROTO_ZIGBEE (O-QPSK)                                         */
    uint8_t  reserved;
    float    cfo_hz, phase0, amp;   /* carrier offset, initial phase (rad), amplitude                                     */
} snrx_tx_burst_t;                  /* 32 bytes */

/* Writes n_steps * 24 cf32 samples of a 96 Msps capture (centre 2440 MHz) to iq_out (device pointer if out_is_device,
 * else host).  bins[n_bins]: filterbank bins in use (n_bins <= 48); taps[384]: the synthesis prototype (gain 24);
 * gauss[16]: Gaussian taps of the GFSK modulator; sigma: noise standard deviation per I / Q component (0 = none). */
int  snrx_synth_wideband(int device, const snrx_tx_burst_t* bursts, uint32_t n_bursts, const uint8_t* data, uint64_t n_data,
                         const int32_t* bins, uint32_t n_bins, const float* taps, const double* gauss, uint64_t n_steps,
                         float sigma, uint64_t seed, float* iq_out, int out_is_device);

int  snrx_set_channel(snrx_t* h, int channel);           /* NB modes */
int  snrx_set_stream(snrx_t* h, void* cuda_stream);       /* run on a caller stream */
int  snrx_sync(snrx_t* h);
int  snrx_stats(snrx_t* h, snrx_stats_t* s);
int  snrx_debug_stage(snrx_t* h, int stage, void* out, uint64_t cap_bytes, uint64_t* n_bytes);
/* Test hook: queue a batch as snrx_process does, but with the BLE slicer bit streams given instead of computed from a
 * capture. words: host memory in the SNRX_STAGE_BLE_BITS layout [n_captures][BLE channels][bits_words_for(n_out)],
 * n_out = n_samples / decimation. The back end, snrx_poll and every call on the polled batch (snrx_ble_aux, snrx_ble_coded,
 * snrx_ble_follow, summaries) then behave as if the channelizer had produced these words.  bits_words_for(n) =
 * 4 lead words + ceil(n / 32) + 64 tail words; bit (m & 31) of word 4 + (m >> 5) is the decision of channel sample m.
 * shard: as in snrx_process (pre_samples and body_samples in input samples).  SNRX_EINVAL for a NULL words, a mode with
 * an 802.15.4 receiver, an engine created with SNRX_F_RF_METRICS or SNRX_F_KEEP_STREAMS (there is no input or channel
 * stream), a wideband n_samples that is not a multiple of 24, or a set bit in the lead words or at a sample >= n_out (the
 * front end never writes one); SNRX_ERANGE and SNRX_ESTATE as snrx_process. */
int snrx_debug_process_bits(snrx_t* h, const uint32_t* words, uint32_t n_captures, uint64_t n_samples,
                            const snrx_shard_t* shard);

/* prototype low-pass of the wideband channelizer (taps = 384 or 768 doubles) */
int  snrx_pfb_prototype(int mode, uint32_t taps, double* out);

/* pinned host staging for callers that want full PCIe rate */
int  snrx_host_alloc(void** p, uint64_t bytes);
int  snrx_host_free(void* p);

/* channel plan helpers (btle_rx.c:932-948; top_block.py:56,94-96) */
int  snrx_ble_channel_mhz(int channel);          /* 37->2402 ... ; <0 on error */
int  snrx_zigbee_channel_mhz(int channel);       /* 11->2405 ... 26->2480      */
int  snrx_ble_channel_bin(int channel);          /* PFB bin (0..95) of a BLE channel  */
int  snrx_zigbee_channel_bin(int channel);

#ifdef __cplusplus
}
#endif
#endif /* SNOUTRX_H */
