// snrx.cu -- C ABI of libsnoutrx.so (include/snoutrx.h) and the host-side orchestration of the
// receive pipelines.  All signal processing happens in the CUDA kernels of this directory; there
// is no CPU implementation behind this interface (no device -> SNRX_ENODEV).
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#ifndef SNRX_LANES
#define SNRX_LANES 2
#endif
#include "ble_adv.cuh"
#include "ble_aux.cuh"
#include "ble_coded.cuh"
#include "ble_sync.cuh"
#include "ble_bis.cuh"
#include "ble_back.cuh"
#include "ble_conn.cuh"
#include "ble_front.cuh"
#include "common.cuh"
#include "pfb.cuh"
#include "pfb_taps.h"
#include "scan.cuh"
#include "zb.cuh"
#include "pfb_zb.cuh"
#include "zb_mac.cuh"
#include "synth.cuh"
#include "frame_rf.cuh"

using namespace snrx;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
};

}  // namespace

// One "lane" per output slot: a complete working set with its own stream, so that the latency-bound tail of
// batch i (search, decode, resolve, export) overlaps the FP32-bound front end of batch i+1.
// Batches that can be queued at once (lanes).  MEASURED (round 2, B200, resident 0.98-s BLE capture, tools/ab_serial.py):
// one batch at a time: channelizer 0.328 ms, whole batch 0.58 ms | two queued: 0.405 ms per step (channelizer 0.39 ms next
// to the other lane's back end) | three queued (-DSNRX_LANES=3): 0.399 ms.  The step is not waiting for the host or for a
// free lane: the back end's kernels (access-address search 39 us, fill 27 us, resolve 37 us, decode 13 us, scans) take
// real SM time from the next channelizer, so a third working set buys 1.5 % and stays off.
constexpr int kLanes = SNRX_LANES;

struct Lane {
    cudaStream_t stream = nullptr;      // front end (channelizer / slicer): low priority, fills the machine
    cudaStream_t tail = nullptr;        // everything after it: high priority, so its small latency-bound kernels are
                                        // dispatched ahead of the other lane's queued channelizer tiles
    snrx_frame_t* frames = nullptr;     // pinned + mapped host copy, frame_cap records
    snrx_frame_t* d_frames = nullptr;   // device list the kernels of the current batch write: one of d_frames_buf, alternating,
    snrx_frame_t* d_frames_buf[2] = {nullptr, nullptr};   // so a polled batch's list stays valid for two further snrx_process calls
    uint32_t uses = 0;
    uint32_t* totals = nullptr;         // pinned: [0] BLE frames [1] candidates [2] Zigbee frames
    uint32_t* d_totals = nullptr;       // device: same layout; [5] CRC-ok frames, [6] arrival counter of k_export_frames' CTAs
    cudaEvent_t ev_start = nullptr, ev_front0 = nullptr, ev_front = nullptr, ev_done = nullptr, ev_in = nullptr;
    cudaEvent_t ev_handoff = nullptr;
    snrx_frame_rf_t* d_rf = nullptr;     // radio metrics the current batch writes (SNRX_F_RF_METRICS): one of d_rf_buf, alternating
    snrx_frame_rf_t* d_rf_buf[2] = {nullptr, nullptr};   // with d_frames_buf, so a polled batch's records outlive the next batch
    bool pending = false, done = false;
    uint32_t caps = 0, n_out = 0, n_frames = 0; uint64_t n_in = 0; int launches = 0;
    // BLE working set
    float2* d_x = nullptr; size_t d_x_bytes = 0;          // staging of host input / cf32 image of sc8 input
    int8_t* d_x8 = nullptr; size_t d_x8_bytes = 0;        // staging of sc8 host input
    uint32_t* d_bits = nullptr; size_t d_bits_bytes = 0;
    uint32_t* d_hits = nullptr;                            // access-address hit masks, same layout as d_bits
    uint32_t *d_counts = nullptr, *d_offsets = nullptr, *d_scratch = nullptr;
    uint32_t *d_wcounts = nullptr, *d_woffsets = nullptr;
    Cand* d_cands = nullptr;
    Dec* d_decs = nullptr;
    int8_t* d_q8 = nullptr; size_t d_q8_bytes = 0;
    float2* d_cf = nullptr; size_t d_cf_bytes = 0;
    ZbState zb;
    std::vector<cudaEvent_t> ev_chunks;
    // the BLE back-end parameters of the lane's last batch (snrx_ble_follow searches its bit streams again)
    BleParams last_p{}; BitsLayout last_lay{}; bool last_ble = false;
};

struct snrx_handle {
    snrx_config_t cfg{};
    int device = 0;
    cudaStream_t user_stream = nullptr;  // stream the caller produces device input on (snrx_set_stream), or null
    cudaStream_t copy_stream = nullptr;  // H2D staging
    // advertising analytics (SURVEY 8f N1), allocated by the first snrx_ble_adv_summary
    cudaStream_t adv_stream = nullptr;
    snrx_adv_t* d_adv = nullptr;
    snrx_zbmac_t* d_zbmac = nullptr;
    snrx_conn_t* d_conn = nullptr; uint32_t *d_conn_flags = nullptr, *d_conn_offsets = nullptr, *d_conn_scratch = nullptr;
    snrx_frame_t* d_follow = nullptr;    // frames of snrx_ble_follow
    // the lists of snrx_ble_aux and snrx_ble_coded (max_frames entries each), allocated by their first call; and what the
    // pointer rounds of both share, allocated by the first of either: flags / offsets / scan scratch of a round and the
    // whitening sequences continued to 260 bytes.  Neither list outlives its call (each is copied out before it returns).
    snrx_ble_aux_t* d_aux = nullptr;
    snrx_ble_coded_t* d_coded = nullptr;
    // snrx_ble_periodic: its trains and its list (max_frames entries each), allocated by its first call; it builds the aux
    // list into d_aux first, and its scans reuse the round buffers once the rounds are done
    snrx::SyncTrain* d_sync_trains = nullptr;
    snrx_ble_sync_t* d_sync = nullptr;
    // snrx_ble_bis: its BIGs and its list (max_frames entries each), allocated by its first call; it builds the periodic list
    // into d_sync first
    snrx::BigGroup* d_bigs = nullptr;
    snrx_ble_bis_t* d_bis = nullptr;
    uint32_t *d_round_flags = nullptr, *d_round_offsets = nullptr, *d_round_scratch = nullptr;
    uint8_t* d_aux_whiten = nullptr;
    snrx::DevSlot* d_devtab = nullptr;
    snrx_device_t* d_devout = nullptr;
    uint32_t* d_adv_counters = nullptr;   // [0] records summarised (BLE), [1] new devices, [2] dropped (table full), [3] export count
    uint32_t dev_count = 0, dev_dropped = 0;
    Lane lane[kLanes];
    uint64_t seq_process = 0, seq_poll = 0;
    // frame exchange (snrx_exchange_*): receive area of this engine and the peers' areas mapped through CUDA IPC
    struct {
        bool connected = false;
        uint32_t rank = 0, world = 1, cap = 0;
        unsigned char* d_recv = nullptr;                       // [world][SNRX_XCHG_SLOTS][1 + cap] records
        unsigned char* peer[SNRX_XCHG_MAX_WORLD] = {nullptr};  // peer[r] = rank r's receive area (peer[rank] = d_recv)
        uint64_t* h_hdr = nullptr;                             // pinned: world x {count, batch}
        cudaStream_t stream = nullptr;
    } xchg;
    int sm_count = 148;
    std::string err;

    // geometry
    bool wideband = false, has_ble = false, has_zb = false;
    int decim = 1;
    uint32_t n_ble_ch = 0, n_zb_ch = 0;
    uint64_t max_in = 0;                 // input samples per capture
    uint32_t max_caps = 1;
    uint32_t max_out = 0;                // channel-rate samples per capture
    uint32_t wpp = 0;                    // words per (capture, channel) bit stream
    uint32_t n_chunks = 0;               // aa-search chunks (32 words) per bit stream
    uint32_t max_windows = 0;
    uint32_t cand_cap = 0, frame_cap = 0;
    int pfb_nt = 16;

    // constants on the device
    uint32_t *d_crc_tab = nullptr, *d_whiten = nullptr;
    int32_t* d_ble_channels = nullptr;
    float *d_taps_rho = nullptr, *d_taps_flat = nullptr, *d_taps_pass = nullptr;
    float* d_rf_taps_zb = nullptr;       // 802.15.4 prototype in tap order (k_frame_rf, wideband modes with 802.15.4 channels)
    double* d_rf_gauss = nullptr;        // Gaussian taps of the GFSK reference (k_frame_rf)

    // last batch
    bool batch_valid = false;
    int last_lane = 0;
    int polled_lane = -1;                // lane of the batch most recently retired by snrx_poll / snrx_poll_view
    const snrx_frame_t* polled_frames_dev = nullptr;   // its device frame list
    const snrx_frame_rf_t* polled_rf_dev = nullptr;    // its radio metrics (SNRX_F_RF_METRICS)
    uint32_t b_caps = 0; uint64_t b_n_in = 0; uint32_t b_n_out = 0;
    snrx_stats_t stats{};
    int launches = 0;
};

namespace {

thread_local std::string g_err;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char b__[512];                                                                         \
            snprintf(b__, sizeof b__, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            if (h) h->err = b__; else g_err = b__;                                                 \
            return e__ == cudaErrorMemoryAllocation ? SNRX_ENOMEM : SNRX_ECUDA;                    \
        }                                                                                          \
    } while (0)

int fail(snrx_handle* h, int code, const char* msg) {
    if (h) h->err = msg; else g_err = msg;
    return code;
}

// ---- BLE tables, built from their definitions --------------------------------------------------
// CRC-24 (x^24+x^10+x^9+x^6+x^4+x^3+x+1) processed LSB first: reflected polynomial 0xDA6000.
// Equals crc_table[] of btle_rx.c:897-930 (tests/test_oracle_ble.py compares via the oracle).
void make_crc_table(uint32_t* t) {
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t r = i;
        for (int k = 0; k < 8; k++) r = (r & 1u) ? (r >> 1) ^ 0xDA6000u : (r >> 1);
        t[i] = r;
    }
}
// Whitening LFSR x^7+x^4+1, register = 1 | channel MSB first (Core spec Vol 6 Part B 3.2): the first n bytes of a channel's
// sequence, LSB first.
void make_whiten_bytes(int ch, uint8_t* bytes, int n) {
    unsigned reg = 0;                           // bit p = register position p
    reg |= 1u;
    for (int k = 0; k < 6; k++) reg |= ((unsigned)(ch >> (5 - k)) & 1u) << (1 + k);
    for (int i = 0; i < n; i++) {
        uint8_t v = 0;
        for (int b = 0; b < 8; b++) {
            unsigned out = (reg >> 6) & 1u;
            v |= (uint8_t)(out << b);
            reg = ((reg << 1) & 0x7Fu) | out;
            reg ^= out << 4;
        }
        bytes[i] = v;
    }
}
// 42 bytes per channel packed little-endian into 11 words.  Equals scramble_table.h.
void make_whiten_table(uint32_t* w /*[40][11]*/) {
    for (int ch = 0; ch < 40; ch++) {
        uint8_t bytes[44] = {0};
        make_whiten_bytes(ch, bytes, 42);
        for (int c = 0; c < 11; c++)
            w[ch * 11 + c] = (uint32_t)bytes[4 * c] | ((uint32_t)bytes[4 * c + 1] << 8) |
                             ((uint32_t)bytes[4 * c + 2] << 16) | ((uint32_t)bytes[4 * c + 3] << 24);
    }
}
// crc_init_reorder(), btle_rx.c:1801-1825: byte swap then 24-bit bit reversal
uint32_t crc_init_internal(uint32_t k) { return crc_seed_of(k); }

template <class T>
int dev_alloc(snrx_handle* h, T** p, size_t count) {
    CK(cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T)));
    return SNRX_OK;
}

uint32_t div_up(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

int grid_for(snrx_handle* h, uint64_t items, int per_block, int blocks_per_sm) {
    uint64_t need = (items + per_block - 1) / per_block;
    uint64_t cap = (uint64_t)h->sm_count * blocks_per_sm;
    return (int)std::max<uint64_t>(1, std::min(need, cap));
}

}  // namespace

static AaTables aa_tables_of(const BleParams& p) {
    const int z = aa_virtual_bits(p.aa, p.aa_mask);
    return make_aa_tables(p.aa, p.aa_mask & ~((1u << z) - 1u));
}

template <int NT>
static int pfb_ble_go(snrx_handle* h, const PfbBleArgs* a, cudaStream_t st, uint32_t caps) {
    using B = PfbBleGeom<NT>;
    if (!a) {
        CK(cudaFuncSetAttribute(k_pfb_ble<NT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B::kSmemBytes));
        CK(cudaFuncSetAttribute(k_pfb_ble<NT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B::kSmemBytes));
        CK(cudaFuncSetAttribute(k_pfb_ble<NT, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        return SNRX_OK;
    }
    if (a->n_tiles <= 0) return SNRX_OK;
    PfbBleArgs b = *a;
    b.n_caps = (int32_t)caps;
    const dim3 grid((unsigned)b.n_tiles, caps);                 // x: tiles, y: captures (snrx_create bounds max_captures by 65535)
    if (h->cfg.flags & SNRX_F_KEEP_STREAMS) k_pfb_ble<NT, true><<<grid, B::kThreads, B::kSmemBytes, st>>>(b);
    else k_pfb_ble<NT, false><<<grid, B::kThreads, B::kSmemBytes, st>>>(b);
    h->launches++;
    return SNRX_OK;
}
static int pfb_ble_dispatch(snrx_handle* h, const PfbBleArgs* a, cudaStream_t st, uint32_t caps) {
    switch (h->pfb_nt) {
        case 16: return pfb_ble_go<16>(h, a, st, caps);
        case 32: return pfb_ble_go<32>(h, a, st, caps);
    }
    return fail(h, SNRX_EINVAL, "no channelizer instance for this configuration");
}
static int ble_tile_stride(const snrx_handle* h) { return h->wideband ? PfbBleGeom<16>::kStride : kTileT; }

// where k_export_frames pushes a batch for the other engines of the node (snrx_exchange_*)
struct ExportXchg {
    unsigned char* peer[SNRX_XCHG_MAX_WORLD];   // receive areas, [src rank][slot][1 + cap] records each
    uint32_t world, rank, cap, slot;            // world = 0: not connected
};
__device__ __forceinline__ uint4* xchg_slot(const ExportXchg& x, uint32_t p) {
    return reinterpret_cast<uint4*>(x.peer[p] + ((size_t)x.rank * SNRX_XCHG_SLOTS + x.slot) * ((size_t)x.cap + 1) * sizeof(snrx_frame_t));
}

// device frame list -> host-mapped pinned memory, fully coalesced 16-byte stores; publishes the totals; and, when the
// engine is connected to its peers, stores the records (only the 16-byte pieces a record uses: 28 bytes of fields + len
// bytes of payload) and then the {count, batch} header into this rank's slot in every rank's receive area -- the frame
// all-gather of the path as plain stores over NVLink, ordered by a system-scope fence before the header goes out.
__global__ void __launch_bounds__(256) k_export_frames(const snrx_frame_t* __restrict__ src, uint32_t* __restrict__ totals_dev,
                                                       snrx_frame_t* __restrict__ dst_host, uint32_t* __restrict__ totals_host,
                                                       uint32_t frame_cap, unsigned long long batch_no, const ExportXchg x) {
    uint32_t n = totals_dev[0] + totals_dev[2];
    if (n > frame_cap) n = frame_cap;                      // few CTAs: this kernel is PCIe bound and must leave the SMs to the other lane
    if (blockIdx.x == 0 && threadIdx.x == 0) {             // header in front of the device list (see the allocation)
        unsigned long long* hdr = reinterpret_cast<unsigned long long*>(const_cast<snrx_frame_t*>(src) - 1);
        hdr[0] = n; hdr[1] = batch_no;
    }
    constexpr uint32_t kPieces = sizeof(snrx_frame_t) / 16;
    const size_t n16 = (size_t)n * kPieces;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst_host);
    uint32_t ok = 0;
    const uint32_t m = x.world ? min(n, x.cap) : 0u;       // world = 0: the engine is not connected to any peer
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = s4[i];
        d4[i] = v;
        const uint32_t rec = (uint32_t)(i / kPieces), k = (uint32_t)(i - (size_t)rec * kPieces);
        if (k == 1) ok += (v.x >> 24) & 1u;                // piece 1 = bytes 16..31: channel, proto, crc_ok, lqi, phase, len, access_addr, bytes[0..3]
        if (rec < m) {
            const uint4 h1 = k == 1 ? v : s4[(size_t)rec * kPieces + 1];
            const uint32_t used = (28u + (h1.y >> 16) + 15u) >> 4;
            if (k < used) {
                for (uint32_t p = 0; p < x.world; p++) xchg_slot(x, p)[(size_t)(rec + 1) * kPieces + k] = v;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ok += __shfl_xor_sync(0xffffffffu, ok, o);
    if ((threadIdx.x & 31) == 0 && ok) atomicAdd(totals_dev + 5, ok);
    // the last CTA to arrive publishes: every store above is ordered before it by the fences
    __shared__ uint32_t ticket;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) ticket = atomicAdd(totals_dev + 6, 1u);
    __syncthreads();
    if (ticket != gridDim.x - 1) return;
    __threadfence_system();
    if (threadIdx.x < 8) totals_host[threadIdx.x] = ((volatile uint32_t*)totals_dev)[threadIdx.x];
    if (threadIdx.x < x.world) {
        const uint4 hdr = make_uint4(n, 0u, (uint32_t)batch_no, (uint32_t)(batch_no >> 32));
        *xchg_slot(x, threadIdx.x) = hdr;                  // {uint64 count, uint64 batch}: 16 bytes, one store
    }
}

// Interleaved signed 8-bit I,Q (the HackRF transfer format the reference consumes: IQ_TYPE int8_t, btle_rx.c:204,
// filled by rx_callback btle_rx.c:489-498) -> cf32 with x = q / 128, exact in FP32.  One sample pair per thread:
// 4-byte loads and 16-byte stores, both coalesced.  n = samples per capture, strides in samples.
__global__ void __launch_bounds__(256) k_sc8_to_cf32(const int8_t* __restrict__ src, uint64_t src_stride, float2* __restrict__ dst,
                                                     uint64_t dst_stride, uint64_t n, uint32_t n_captures) {
    const uint64_t pairs = (n + 1) / 2;
    const uint64_t total = pairs * n_captures;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t c = i / pairs, p = i - c * pairs;
        const int8_t* s = src + 2 * (c * src_stride + 2 * p);
        float2* d = dst + c * dst_stride + 2 * p;
        if (2 * p + 1 < n) {
            const char4 q = __ldcs(reinterpret_cast<const char4*>(s));
            __stcs(reinterpret_cast<float4*>(d), make_float4(q.x * 0.0078125f, q.y * 0.0078125f, q.z * 0.0078125f, q.w * 0.0078125f));
        } else {
            d[0] = make_float2(s[0] * 0.0078125f, s[1] * 0.0078125f);
        }
    }
}

extern "C" {

int snrx_abi_version(void) { return SNRX_ABI_VERSION; }

const char* snrx_strerror(int code) {
    switch (code) {
        case SNRX_OK: return "ok";
        case SNRX_EINVAL: return "invalid argument or configuration";
        case SNRX_ENODEV: return "no usable CUDA device (libsnoutrx has no CPU fallback)";
        case SNRX_ENOMEM: return "out of host or device memory";
        case SNRX_ECUDA: return "CUDA runtime error";
        case SNRX_ERANGE: return "input exceeds the configured capacity";
        case SNRX_EOVERFLOW: return "more candidates or frames than the configured capacity";
        case SNRX_ESTATE: return "call out of sequence";
        default: return "unknown error";
    }
}

const char* snrx_last_error(snrx_t* h) { return h ? h->err.c_str() : g_err.c_str(); }

int snrx_device_count(int* n) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (n) *n = (e == cudaSuccess) ? c : 0;
    return (e == cudaSuccess && c > 0) ? SNRX_OK : SNRX_ENODEV;
}

int snrx_ble_channel_mhz(int ch) { return ble_channel_mhz(ch); }
int snrx_zigbee_channel_mhz(int ch) { return zb_channel_mhz(ch); }
int snrx_ble_channel_bin(int ch) { return pfb_bin_of_mhz(ble_channel_mhz(ch)); }
int snrx_zigbee_channel_bin(int ch) { return pfb_bin_of_mhz(zb_channel_mhz(ch)); }

int snrx_pfb_prototype(int mode, uint32_t taps, double* out) {
    const bool zb = (mode == SNRX_MODE_ZB_WB16);
    const double* src = nullptr;
    if (taps == 384) src = zb ? SNRX_PFB_ZB_384 : SNRX_PFB_BLE_384;
    else if (taps == 768) src = zb ? SNRX_PFB_ZB_768 : SNRX_PFB_BLE_768;
    else return SNRX_EINVAL;
    memcpy(out, src, sizeof(double) * taps);
    return SNRX_OK;
}

void snrx_destroy(snrx_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (auto& ln : h->lane) { if (ln.stream) cudaStreamSynchronize(ln.stream); if (ln.tail) cudaStreamSynchronize(ln.tail); }
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    void* bufs[] = {h->d_crc_tab, h->d_whiten, h->d_ble_channels, h->d_taps_rho, h->d_taps_flat, h->d_taps_pass, h->d_rf_taps_zb,
                    h->d_rf_gauss};
    for (void* b : bufs) if (b) cudaFree(b);
    for (auto& ln : h->lane) {
        void* lb[] = {ln.d_x, ln.d_x8, ln.d_bits, ln.d_hits, ln.d_counts, ln.d_offsets, ln.d_scratch, ln.d_wcounts, ln.d_woffsets,
                      ln.d_cands, ln.d_decs, ln.d_totals, ln.d_q8, ln.d_cf,
                      ln.d_frames_buf[0] ? ln.d_frames_buf[0] - 1 : nullptr, ln.d_frames_buf[1] ? ln.d_frames_buf[1] - 1 : nullptr,
                      ln.d_rf_buf[0], ln.d_rf_buf[1]};
        for (void* b : lb) if (b) cudaFree(b);
        zb_free(ln.zb);
        if (ln.frames) cudaFreeHost(ln.frames);
        if (ln.totals) cudaFreeHost(ln.totals);
        for (cudaEvent_t e : {ln.ev_start, ln.ev_front0, ln.ev_front, ln.ev_done, ln.ev_in, ln.ev_handoff}) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : ln.ev_chunks) cudaEventDestroy(e);
        if (ln.stream) cudaStreamDestroy(ln.stream);
        if (ln.tail) cudaStreamDestroy(ln.tail);
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->xchg.stream) { cudaStreamSynchronize(h->xchg.stream); cudaStreamDestroy(h->xchg.stream); }
    for (uint32_t r = 0; r < h->xchg.world && r < SNRX_XCHG_MAX_WORLD; r++)
        if (h->xchg.peer[r] && h->xchg.peer[r] != h->xchg.d_recv) cudaIpcCloseMemHandle(h->xchg.peer[r]);
    if (h->xchg.d_recv) cudaFree(h->xchg.d_recv);
    if (h->xchg.h_hdr) cudaFreeHost(h->xchg.h_hdr);
    if (h->adv_stream) { cudaStreamSynchronize(h->adv_stream); cudaStreamDestroy(h->adv_stream); }
    { void* ab[] = {h->d_adv, h->d_zbmac, h->d_conn, h->d_conn_flags, h->d_conn_offsets, h->d_conn_scratch, h->d_follow, h->d_devtab, h->d_devout, h->d_adv_counters,
                    h->d_aux, h->d_coded, h->d_round_flags, h->d_round_offsets, h->d_round_scratch, h->d_aux_whiten,
                    h->d_sync_trains, h->d_sync, h->d_bigs, h->d_bis}; for (void* b : ab) if (b) cudaFree(b); }
    delete h;
}

int snrx_create(snrx_t** out, const snrx_config_t* cfg) {
    snrx_handle* h = nullptr;
    if (!out || !cfg) return fail(nullptr, SNRX_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != SNRX_ABI_VERSION) return fail(nullptr, SNRX_EINVAL, "abi_version mismatch");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(nullptr, SNRX_ENODEV, "no CUDA device: libsnoutrx has no CPU path");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, SNRX_ENODEV, "device ordinal out of range");
    h = new (std::nothrow) snrx_handle();
    if (!h) return fail(nullptr, SNRX_ENOMEM, "host allocation failed");
    h->cfg = *cfg;
    h->device = cfg->device;
#define CKD(call) do { int r__ = (call); if (r__ != SNRX_OK) return r__; } while (0)
    auto body = [&]() -> int {
        CK(cudaSetDevice(h->device));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, h->device));
        h->sm_count = prop.multiProcessorCount;
        if (prop.major < 10) return fail(h, SNRX_ENODEV, "libsnoutrx is built for sm_100a (B200) only");
        CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));

        snrx_config_t& c = h->cfg;
        switch (c.mode) {
            case SNRX_MODE_BLE_NB: h->has_ble = true; h->n_ble_ch = 1; h->decim = 1; break;
            case SNRX_MODE_ZB_NB: h->has_zb = true; h->n_zb_ch = 1; h->decim = 1; break;
            case SNRX_MODE_BLE_WB40: h->has_ble = true; h->wideband = true; h->n_ble_ch = 40; h->decim = kPfbD; break;
            case SNRX_MODE_ZB_WB16: h->has_zb = true; h->wideband = true; h->n_zb_ch = 16; h->decim = kPfbD; break;
            case SNRX_MODE_MIXED_WB56:
                h->has_ble = h->has_zb = true; h->wideband = true; h->n_ble_ch = 40; h->n_zb_ch = 16; h->decim = kPfbD; break;
            default: return fail(h, SNRX_EINVAL, "unknown mode");
        }
        if (c.access_addr == 0 && c.crc_init == 0) { c.access_addr = 0x8E89BED6u; c.crc_init = 0x555555u; }
        if (c.zb_threshold <= 0) c.zb_threshold = 10;
        if (c.quant_scale <= 0.0f) c.quant_scale = h->wideband ? 100.0f : 128.0f;
        if (c.max_captures == 0) c.max_captures = 1;
        if (h->wideband && c.max_captures > 65535u) return fail(h, SNRX_ERANGE, "wideband engines take at most 65535 captures per batch (the captures are the y dimension of the channelizer grids)");
        if (c.max_samples == 0) c.max_samples = h->wideband ? 96000000ull : 10000000ull;
        if (c.max_frames == 0) c.max_frames = 1u << 17;
        if (c.zb_segment == 0) c.zb_segment = SNRX_ZB_SEGMENT_DEFAULT;
        if (c.zb_prehalo == 0) c.zb_prehalo = SNRX_ZB_PREHALO_DEFAULT;
        if (c.pfb_taps == 0) c.pfb_taps = 384;
        if (c.pfb_taps != 384 && c.pfb_taps != 768) return fail(h, SNRX_EINVAL, "pfb_taps must be 384 or 768");
        h->pfb_nt = (int)c.pfb_taps / 24;
        if (h->has_ble && !h->wideband && (c.channel < 0 || c.channel > 39)) return fail(h, SNRX_EINVAL, "BLE channel 0..39");
        if (h->has_zb && !h->wideband && (c.channel < 11 || c.channel > 26)) return fail(h, SNRX_EINVAL, "802.15.4 channel 11..26");
        // With no compared 1 bit, runs of zero decisions match the address: btle_rx.c then "finds" a frame at every search origin,
        // in the zero samples past the end of a capture too, where the sliding correlation (k_aa_search) has no start positions.
        if (h->has_ble && (c.access_addr & (c.access_mask ? c.access_mask : 0xFFFFFFFFu)) == 0u)
            return fail(h, SNRX_EINVAL, "BLE access_addr & access_mask must have a bit set");
        if (h->wideband && (c.max_samples % (uint64_t)(kPfbD * 2)) != 0) c.max_samples += (kPfbD * 2) - c.max_samples % (kPfbD * 2);
        h->max_in = c.max_samples;
        h->max_caps = c.max_captures;
        h->max_out = (uint32_t)(h->max_in / h->decim);
        h->frame_cap = c.max_frames;
        h->cand_cap = std::max<uint32_t>(1u << 16, 4 * c.max_frames);

        if (h->has_ble) {
            h->wpp = bits_words_for(h->max_out);
            h->n_chunks = div_up(h->wpp, 32);
            h->max_windows = div_up(h->max_out, kWindow);
            uint32_t crc[256], wh[40 * 11];
            make_crc_table(crc);
            make_whiten_table(wh);
            CKD(dev_alloc(h, &h->d_crc_tab, 256));
            CKD(dev_alloc(h, &h->d_whiten, 40 * 11));
            CK(cudaMemcpy(h->d_crc_tab, crc, sizeof crc, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->d_whiten, wh, sizeof wh, cudaMemcpyHostToDevice));
            int32_t chans[40];
            for (int i = 0; i < 40; i++) chans[i] = h->wideband ? i : c.channel;
            CKD(dev_alloc(h, &h->d_ble_channels, 40));
            CK(cudaMemcpy(h->d_ble_channels, chans, sizeof chans, cudaMemcpyHostToDevice));
            if (h->wideband) {
                const int L = (int)c.pfb_taps, NT = h->pfb_nt;
                const double* proto = (L == 384) ? SNRX_PFB_BLE_384 : SNRX_PFB_BLE_768;
                std::vector<float> flat(L), rho(L);
                for (int n = 0; n < L; n++) flat[n] = (float)proto[n];
                for (int r = 0; r < 24; r++) for (int d = 0; d < NT; d++) rho[r * NT + d] = flat[r + 24 * d];
                CKD(dev_alloc(h, &h->d_taps_rho, L));
                CKD(dev_alloc(h, &h->d_taps_flat, L));
                CK(cudaMemcpy(h->d_taps_rho, rho.data(), sizeof(float) * L, cudaMemcpyHostToDevice));
                CK(cudaMemcpy(h->d_taps_flat, flat.data(), sizeof(float) * L, cudaMemcpyHostToDevice));
                // per-pass layout of k_pfb_ble: [gi][d4][rl][4] = h[rho + 24 (4 d4 + k)], rho = gi + 3 rl
                std::vector<float> pass(L);
                for (int gi = 0; gi < 3; gi++) for (int d4 = 0; d4 < NT / 4; d4++) for (int rl = 0; rl < 8; rl++) for (int k = 0; k < 4; k++)
                    pass[((gi * (NT / 4) + d4) * 8 + rl) * 4 + k] = flat[(gi + 3 * rl) + 24 * (4 * d4 + k)];
                CKD(dev_alloc(h, &h->d_taps_pass, L));
                CK(cudaMemcpy(h->d_taps_pass, pass.data(), sizeof(float) * L, cudaMemcpyHostToDevice));
                int r = pfb_ble_dispatch(h, nullptr, nullptr, 0);                          // sets the shared-memory attributes
                if (r != SNRX_OK) return r;
            }
        }
        if (c.flags & SNRX_F_RF_METRICS) {
            double g[16];
            rf_gauss_taps(g);
            CKD(dev_alloc(h, &h->d_rf_gauss, 16));
            CK(cudaMemcpy(h->d_rf_gauss, g, sizeof g, cudaMemcpyHostToDevice));
            if (h->has_zb && h->wideband) {
                const double* proto = (c.pfb_taps == 384) ? SNRX_PFB_ZB_384 : SNRX_PFB_ZB_768;
                std::vector<float> flat(c.pfb_taps);
                for (uint32_t n = 0; n < c.pfb_taps; n++) flat[n] = (float)proto[n];
                CKD(dev_alloc(h, &h->d_rf_taps_zb, c.pfb_taps));
                CK(cudaMemcpy(h->d_rf_taps_zb, flat.data(), sizeof(float) * c.pfb_taps, cudaMemcpyHostToDevice));
            }
            CK(cudaFuncSetAttribute(k_frame_rf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rf_smem_bytes(32)));
        }
        for (auto& ln : h->lane) {
            int prio_lo = 0, prio_hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            CK(cudaStreamCreateWithPriority(&ln.stream, cudaStreamNonBlocking, prio_lo));
            CK(cudaStreamCreateWithPriority(&ln.tail, cudaStreamNonBlocking, prio_hi));
            CK(cudaEventCreateWithFlags(&ln.ev_handoff, cudaEventDisableTiming));
            CK(cudaHostAlloc((void**)&ln.frames, sizeof(snrx_frame_t) * (size_t)h->frame_cap, cudaHostAllocMapped));
            CK(cudaHostAlloc((void**)&ln.totals, 8 * sizeof(uint32_t), cudaHostAllocMapped));
            CK(cudaEventCreate(&ln.ev_start));
            CK(cudaEventCreate(&ln.ev_front0));
            CK(cudaEventCreate(&ln.ev_front));
            CK(cudaEventCreate(&ln.ev_done));
            CK(cudaEventCreateWithFlags(&ln.ev_in, cudaEventDisableTiming));
            // one record of room in front of every list: k_export_frames writes {uint64 count, uint64 batch number} there,
            // so [header | records] can leave the GPU as one block (dist.PeerGather)
            for (auto& fb : ln.d_frames_buf) { CK(cudaMalloc((void**)&fb, sizeof(snrx_frame_t) * ((size_t)h->frame_cap + 1))); fb += 1; }
            ln.d_frames = ln.d_frames_buf[0];
            if (c.flags & SNRX_F_RF_METRICS) {
                for (auto& rb : ln.d_rf_buf) CKD(dev_alloc(h, &rb, h->frame_cap));
                ln.d_rf = ln.d_rf_buf[0];
            }
            CKD(dev_alloc(h, &ln.d_totals, 8));
            CK(cudaMemset(ln.d_totals, 0, 8 * sizeof(uint32_t)));
            if (h->has_ble) {
                ln.d_bits_bytes = (size_t)h->max_caps * h->n_ble_ch * h->wpp * sizeof(uint32_t);
                CK(cudaMalloc((void**)&ln.d_bits, ln.d_bits_bytes));
                CK(cudaMalloc((void**)&ln.d_hits, ln.d_bits_bytes));
                const size_t aa_items = (size_t)h->max_caps * h->n_ble_ch * h->n_chunks;
                const size_t w_items = (size_t)h->max_caps * h->n_ble_ch * h->max_windows;
                CKD(dev_alloc(h, &ln.d_counts, aa_items + 1));
                CKD(dev_alloc(h, &ln.d_offsets, aa_items + 1));
                CKD(dev_alloc(h, &ln.d_wcounts, w_items + 1));
                CKD(dev_alloc(h, &ln.d_woffsets, w_items + 1));
                CKD(dev_alloc(h, &ln.d_scratch, scan_scratch_items(std::max(aa_items, w_items))));
                CKD(dev_alloc(h, &ln.d_cands, h->cand_cap));
                CKD(dev_alloc(h, &ln.d_decs, h->cand_cap));
                if (c.flags & SNRX_F_KEEP_STREAMS) {
                    ln.d_q8_bytes = (size_t)h->max_caps * h->n_ble_ch * h->max_out * 2;
                    CK(cudaMalloc((void**)&ln.d_q8, ln.d_q8_bytes));
                    if (h->wideband) {
                        ln.d_cf_bytes = (size_t)h->max_caps * h->n_ble_ch * h->max_out * sizeof(float2);
                        CK(cudaMalloc((void**)&ln.d_cf, ln.d_cf_bytes));
                    }
                }
            }
            if (h->has_zb) {
                int r = zb_create(ln.zb, h->cfg, h->wideband, h->n_zb_ch, h->max_caps, h->max_out, h->sm_count, h->err);
                if (r != SNRX_OK) return r;
                if (h->wideband) {
                    const double* proto = (c.pfb_taps == 384) ? SNRX_PFB_ZB_384 : SNRX_PFB_ZB_768;
                    r = zb_wideband_init(ln.zb, h->cfg, proto, h->max_caps, h->max_out, h->err);
                    if (r != SNRX_OK) return r;
                }
            }
        }
        return SNRX_OK;
    };
    int r = body();
    if (r != SNRX_OK) { g_err = h->err; snrx_destroy(h); return r; }
    *out = h;
    return SNRX_OK;
#undef CKD
}

int snrx_set_stream(snrx_t* h, void* cuda_stream) {
    if (!h) return SNRX_EINVAL;
    h->user_stream = (cudaStream_t)cuda_stream;
    return SNRX_OK;
}

int snrx_set_channel(snrx_t* h, int channel) {
    if (!h) return SNRX_EINVAL;
    if (h->wideband) return fail(h, SNRX_EINVAL, "set_channel applies to the narrow-band modes");
    CK(cudaSetDevice(h->device));
    for (auto& ln : h->lane) CK(cudaStreamSynchronize(ln.tail));         // queued batches keep the channel they were queued with
    if (h->has_ble) {
        if (channel < 0 || channel > 39) return fail(h, SNRX_EINVAL, "BLE channel 0..39");
        int32_t chans[40];
        for (int i = 0; i < 40; i++) chans[i] = channel;
        CK(cudaMemcpy(h->d_ble_channels, chans, sizeof chans, cudaMemcpyHostToDevice));
    } else {
        if (channel < 11 || channel > 26) return fail(h, SNRX_EINVAL, "802.15.4 channel 11..26");
        int32_t chans[16];
        for (int i = 0; i < 16; i++) chans[i] = channel;
        for (auto& ln : h->lane) CK(cudaMemcpy(ln.zb.d_channels, chans, sizeof chans, cudaMemcpyHostToDevice));
    }
    h->cfg.channel = channel;
    return SNRX_OK;
}

int snrx_sync(snrx_t* h) {
    if (!h) return SNRX_EINVAL;
    CK(cudaSetDevice(h->device));
    for (auto& ln : h->lane) { CK(cudaStreamSynchronize(ln.stream)); CK(cudaStreamSynchronize(ln.tail)); }
    return SNRX_OK;
}

// ------------------------------------------------------------------------------------ process
static int launch_ble_front(snrx_handle* h, Lane& ln, const float2* x, uint32_t caps, uint64_t n_in, uint64_t stride,
                            uint32_t n_out, int tile_begin, int tile_end, BitsLayout lay) {
    const bool dbg = (h->cfg.flags & SNRX_F_KEEP_STREAMS) != 0;
    if (h->wideband) {
        PfbBleArgs a;
        a.x = x; a.stride = stride; a.n_in = (int64_t)n_in; a.n_out = (int32_t)n_out;
        a.n_tiles = tile_end - tile_begin;
        a.taps_pass = reinterpret_cast<const float4*>(h->d_taps_pass); a.scale = h->cfg.quant_scale;
        a.bits = ln.d_bits; a.lay = lay; a.dbg_q8 = ln.d_q8; a.dbg_cf = ln.d_cf;
        a.tile0 = tile_begin;
        int r = pfb_ble_dispatch(h, &a, ln.stream, caps);
        if (r != SNRX_OK) return r;
        CK(cudaGetLastError());
        return SNRX_OK;
    } else {
        NbArgs a;
        a.x = x; a.stride = stride; a.n = (int64_t)n_in;
        a.n_groups = (int32_t)div_up(n_in, 128); a.n_captures = caps; a.scale = h->cfg.quant_scale;
        a.bits = ln.d_bits; a.lay = lay; a.dbg_q8 = ln.d_q8;
        const uint32_t per_cap_max = (uint32_t)div_up((uint64_t)a.n_groups, 8);                  // 8 warps per block, one item each
        a.blocks_per_cap = std::max<uint32_t>(1u, std::min<uint32_t>(per_cap_max, (uint32_t)div_up((uint64_t)h->sm_count * 8, caps)));
        const unsigned grid = a.blocks_per_cap * caps;
        if (dbg) k_ble_slice_nb<true><<<grid, 256, 0, ln.stream>>>(a);
        else k_ble_slice_nb<false><<<grid, 256, 0, ln.stream>>>(a);
    }
    h->launches++;
    CK(cudaGetLastError());
    return SNRX_OK;
}

}  // extern "C"

enum { kFmtCf32 = 0, kFmtSc8 = 1 };

// true if no bit is set in the lead words or at a sample >= n_out of any stream ([streams][bits_words_for(n_out)])
static bool bits_outside_clear(const uint32_t* words, uint64_t n_streams, uint32_t n_out) {
    const uint64_t wpp = bits_words_for(n_out);
    const uint32_t body = (n_out + 31) / 32, partial = n_out & 31;
    for (uint64_t st = 0; st < n_streams; st++) {
        const uint32_t* w = words + st * wpp;
        for (uint64_t i = 0; i < wpp; i++) {
            const uint64_t b = i - kBitsLeadWords;                 // body word (wraps for the lead words)
            const uint32_t allowed = b >= body ? 0u : (b + 1 == body && partial ? (1u << partial) - 1u : 0xFFFFFFFFu);
            if (w[i] & ~allowed) return false;
        }
    }
    return true;
}

// The BLE back end over a lane's bit streams, on stream st: access-address search -> scan -> candidate fill -> decode ->
// resolve (count per window) -> scan -> resolve (write) into `frames` (frame_cap records).  snrx_process runs it on the
// batch's streams, snrx_ble_follow again on the polled batch's streams with another address.  The kernels use grid-stride
// loops, so the grids set the speed, not the result: 8 blocks per SM of the grid-limited kernels.  MEASURED
// (tools/ab_serial.py, ms per step with two batches queued): 8 blocks 0.404 | 4 blocks 0.402 | 2 blocks 0.422 | 1 block
// 0.471 -- smaller grids do not give the next batch's channelizer more of the machine, they only stretch the latency-bound
// chain search -> scan -> fill -> decode -> resolve -> export until it no longer fits beside one channelizer launch.
struct BackTotals {
    const uint32_t* frames;       // device: frames the chain found (may exceed frame_cap: the list then holds frame_cap)
    const uint32_t* cands;        // device: access-address candidates (may exceed cand_cap)
};
static int launch_ble_back(snrx_handle* h, Lane& ln, const BleParams& p, const BitsLayout& lay, snrx_frame_t* frames,
                           cudaStream_t st, BackTotals* tot) {
    const uint32_t n_chunks = div_up(lay.words_per_stream, 32);
    const uint32_t aa_items = p.n_captures * h->n_ble_ch * n_chunks;
    const uint32_t w_items = p.n_captures * h->n_ble_ch * (uint32_t)p.n_windows;
    k_aa_search<<<grid_for(h, aa_items, 8, 8), 256, 0, st>>>(ln.d_bits, lay, p, n_chunks, ln.d_counts, ln.d_hits, aa_tables_of(p));
    h->launches += 1 + exclusive_scan(ln.d_counts, aa_items, ln.d_offsets, ln.d_scratch, st);
    k_aa_fill<<<grid_for(h, aa_items, 256, 8), 256, 0, st>>>(ln.d_bits, ln.d_hits, lay, p, n_chunks, ln.d_counts, ln.d_offsets, ln.d_cands, h->cand_cap);
    k_ble_decode<<<h->sm_count * 16, 128, 0, st>>>(ln.d_bits, lay, p, ln.d_offsets + aa_items, h->cand_cap, ln.d_cands,
                                               ln.d_decs, h->d_crc_tab, h->d_whiten, h->d_ble_channels);
    const int g_w = grid_for(h, w_items, 256, 8);
    k_ble_resolve<false><<<g_w, 256, 0, st>>>(ln.d_cands, ln.d_decs, ln.d_offsets, n_chunks, p, ln.d_wcounts, nullptr,
                                             nullptr, 0, h->d_ble_channels, h->cand_cap);
    h->launches += 3 + exclusive_scan(ln.d_wcounts, w_items, ln.d_woffsets, ln.d_scratch, st);
    k_ble_resolve<true><<<g_w, 256, 0, st>>>(ln.d_cands, ln.d_decs, ln.d_offsets, n_chunks, p, ln.d_wcounts, ln.d_woffsets,
                                            frames, h->frame_cap, h->d_ble_channels, h->cand_cap);
    h->launches += 1;
    CK(cudaGetLastError());
    tot->frames = ln.d_woffsets + w_items;
    tot->cands = ln.d_offsets + aa_items;
    return SNRX_OK;
}

// bits != nullptr: snrx_debug_process_bits -- the BLE slicer words are given (host memory, SNRX_STAGE_BLE_BITS layout)
// instead of computed from iq; no input is staged and no front end runs.  Everything from the back end on is shared.
static int process_impl(snrx_t* h, const void* iq, int fmt, uint32_t n_captures, uint64_t n_samples, uint64_t stride_samples,
                        const snrx_shard_t* shard, int is_device_ptr, const uint32_t* bits = nullptr) {
    if (!h || !(iq || bits)) return SNRX_EINVAL;
    if (n_captures == 0 || n_samples == 0) return fail(h, SNRX_EINVAL, "empty batch");
    if (n_captures > h->max_caps || n_samples > h->max_in) return fail(h, SNRX_ERANGE, "batch exceeds max_captures/max_samples");
    if (stride_samples == 0) stride_samples = n_samples;
    if (stride_samples < n_samples) return fail(h, SNRX_EINVAL, "stride smaller than the capture");
    if (!bits && ((((uintptr_t)iq) & 15) || (n_captures > 1 && (stride_samples & 1)))) return fail(h, SNRX_EINVAL, "captures must be 16-byte aligned (even stride)");
    if (h->wideband && (n_samples % kPfbD) != 0) return fail(h, SNRX_EINVAL, "wideband captures must hold a multiple of 24 samples");
    if (bits && !bits_outside_clear(bits, (uint64_t)n_captures * h->n_ble_ch, (uint32_t)(n_samples / h->decim)))
        return fail(h, SNRX_EINVAL, "snrx_debug_process_bits: a bit is set in the lead words or past the capture's last sample");
    CK(cudaSetDevice(h->device));
    const int li = (int)(h->seq_process % kLanes);
    Lane& ln = h->lane[li];
    if (ln.pending) return fail(h, SNRX_ESTATE, "every lane holds a queued batch: snrx_poll the oldest first");
    h->launches = 0;
    // this lane's previous batch (two batches ago) has been polled, hence finished: its buffers are free
    cudaStream_t st = ln.stream;

    const uint32_t n_out = (uint32_t)(n_samples / h->decim);
    uint32_t pre_out = 0, body_out = n_out, first_window = 0, first_capture = 0;
    if (shard) {
        if (shard->pre_samples % (uint64_t)(h->decim * kTileT)) return fail(h, SNRX_EINVAL, "pre_samples must be a multiple of 128 channel samples");
        pre_out = (uint32_t)(shard->pre_samples / h->decim);
        body_out = shard->body_samples ? (uint32_t)(shard->body_samples / h->decim) : n_out - pre_out;
        first_window = shard->first_window;
        first_capture = shard->first_capture_id;
        if ((uint64_t)pre_out + body_out > n_out) return fail(h, SNRX_EINVAL, "shard body exceeds the buffer");
        if (h->has_zb) {
            // the DC tracker is defined on the absolute SNRX_IIR_BLOCK grid with a memory of SNRX_IIR_MEMORY_BLOCKS blocks, the
            // chains on the absolute segment grid: a shard reproduces the whole-capture result only from there on
            const uint32_t seg = h->cfg.zb_segment;
            if ((seg % kWindow) && (kWindow % seg)) return fail(h, SNRX_EINVAL, "Zigbee shards need zb_segment to divide 8192 or be a multiple of it");
            if (pre_out % SNRX_IIR_BLOCK) return fail(h, SNRX_EINVAL, "Zigbee shards: pre_samples must be a multiple of 2048 channel samples");
            if (((uint64_t)first_window * kWindow) % seg) return fail(h, SNRX_EINVAL, "Zigbee shards: the body must start on the segment grid");
            const uint32_t need = (SNRX_IIR_MEMORY_BLOCKS + 1) * SNRX_IIR_BLOCK + h->cfg.zb_prehalo;   // +1: the first block of a
            // buffer holds a discriminator sample without history (and the channelizer start-up), so its end value is off
            // (a buffer that starts at capture sample 0 holds the whole history there is)
            if (first_window != 0 && pre_out < need && (uint64_t)first_window * kWindow != pre_out) return fail(h, SNRX_EINVAL, "Zigbee shards: pre halo shorter than (48 + 1) * 2048 + zb_prehalo channel samples");
        }
    }

    if (shard && (h->cfg.flags & SNRX_F_RF_METRICS) && h->has_ble && h->wideband && h->pfb_nt == 32 && pre_out < 256 &&
        (uint64_t)first_window * kWindow != pre_out)
        return fail(h, SNRX_EINVAL, "radio metrics with 768 taps: a BLE shard that does not start the capture needs a pre halo of >= 256 channel samples");

    if (is_device_ptr && h->user_stream) {          // device input is produced on the caller's stream
        CK(cudaEventRecord(ln.ev_in, h->user_stream));
        CK(cudaStreamWaitEvent(st, ln.ev_in, 0));
    }
    CK(cudaEventRecord(ln.ev_start, st));
    CK(cudaMemsetAsync(ln.d_totals, 0, 8 * sizeof(uint32_t), st));
    if (ln.d_rf_buf[0]) ln.d_rf = ln.d_rf_buf[ln.uses & 1];
    ln.d_frames = ln.d_frames_buf[ln.uses++ & 1];

    // ---- input: cf32 device pointer as is; host pointer staged in chunks overlapped with the front end;
    //      sc8 input (host or device) is expanded to cf32 in ln.d_x by k_sc8_to_cf32, chunk by chunk
    const float2* x = reinterpret_cast<const float2*>(iq);
    uint64_t x_stride = stride_samples;
    const bool staged = !is_device_ptr && !bits;
    const bool sc8 = (fmt == kFmtSc8) && !bits;
    const uint64_t chunk_samples = sc8 ? (8ull << 20) : (4ull << 20);   // 16 MiB (sc8) / 32 MiB (cf32) per copy
    const size_t in_elem = sc8 ? 2 : sizeof(float2);                // bytes per input sample
    if (staged || sc8) {
        x_stride = n_samples + (n_samples & 1);                     // captures stay 16-byte aligned
        const size_t need = (size_t)n_captures * x_stride * sizeof(float2);
        if (need > ln.d_x_bytes) {
            if (ln.d_x) { cudaFree(ln.d_x); ln.d_x = nullptr; ln.d_x_bytes = 0; }
            CK(cudaMalloc((void**)&ln.d_x, need));
            ln.d_x_bytes = need;
        }
        x = ln.d_x;
    }
    if (staged && sc8) {
        const size_t need = (size_t)n_captures * x_stride * 2;
        if (need > ln.d_x8_bytes) {
            if (ln.d_x8) { cudaFree(ln.d_x8); ln.d_x8 = nullptr; ln.d_x8_bytes = 0; }
            CK(cudaMalloc((void**)&ln.d_x8, need));
            ln.d_x8_bytes = need;
        }
    }
    if (sc8 && !staged) {                                           // device sc8: one expansion pass over the batch
        k_sc8_to_cf32<<<h->sm_count * 8, 256, 0, st>>>(reinterpret_cast<const int8_t*>(iq), stride_samples, ln.d_x, x_stride,
                                                       n_samples, n_captures);
        h->launches++;
        CK(cudaGetLastError());
    }

    BitsLayout lay{};
    if (h->has_ble) {
        lay.words_per_stream = bits_words_for(n_out);
        lay.n_channels = h->n_ble_ch;
        const size_t bytes = (size_t)n_captures * h->n_ble_ch * lay.words_per_stream * sizeof(uint32_t);
        if (bits) CK(cudaMemcpyAsync(ln.d_bits, bits, bytes, cudaMemcpyHostToDevice, st));
        else CK(cudaMemsetAsync(ln.d_bits, 0, bytes, st));
    }

    if (staged) {
        CK(cudaEventRecord(ln.ev_front0, st));
        // the copy stream serialises the staging copies of both lanes (one PCIe link anyway)
        size_t ev_i = 0;
        for (uint32_t c = 0; c < n_captures; c++) {
            const char* src = reinterpret_cast<const char*>(iq) + (size_t)c * stride_samples * in_elem;
            char* dst = sc8 ? reinterpret_cast<char*>(ln.d_x8) + (size_t)c * x_stride * in_elem
                            : reinterpret_cast<char*>(ln.d_x + (size_t)c * x_stride);
            int tile_done = 0;
            for (uint64_t off = 0; off < n_samples; off += chunk_samples) {
                const uint64_t len = std::min<uint64_t>(chunk_samples, n_samples - off);
                CK(cudaMemcpyAsync(dst + off * in_elem, src + off * in_elem, len * in_elem, cudaMemcpyHostToDevice, h->copy_stream));
                if (ev_i >= ln.ev_chunks.size()) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ln.ev_chunks.push_back(e); }
                CK(cudaEventRecord(ln.ev_chunks[ev_i], h->copy_stream));
                CK(cudaStreamWaitEvent(st, ln.ev_chunks[ev_i], 0));
                ev_i++;
                if (sc8) {                                          // chunk_samples is even: pairs never straddle chunks
                    k_sc8_to_cf32<<<h->sm_count * 4, 256, 0, st>>>(reinterpret_cast<const int8_t*>(dst) + off * 2, 0,
                                                                   ln.d_x + (size_t)c * x_stride + off, 0, len, 1);
                    h->launches++;
                }
                if (h->has_ble && h->wideband && !h->has_zb && n_captures == 1) {
                    // launch the channelizer on the tiles whose input has fully arrived
                    const uint64_t have = off + len;
                    const bool last = (have == n_samples);
                    const int ts = ble_tile_stride(h);
                    int tile_end = last ? (int)div_up(n_out, ts) : (int)(((int64_t)(have / kPfbD) - (ts + 1)) / ts);
                    if (tile_end > tile_done) {
                        int r = launch_ble_front(h, ln, x, 1, n_samples, x_stride, n_out, tile_done, tile_end, lay);
                        if (r != SNRX_OK) return r;
                        tile_done = tile_end;
                    }
                }
            }
        }
    }

    if (h->has_ble) {
        const bool pipelined = staged && h->wideband && !h->has_zb && n_captures == 1;
        if (!pipelined) {
            CK(cudaEventRecord(ln.ev_front0, st));
            if (!bits) {
                int r = launch_ble_front(h, ln, x, n_captures, n_samples, x_stride, n_out, 0, (int)div_up(n_out, ble_tile_stride(h)), lay);
                if (r != SNRX_OK) return r;
            }
        }
        CK(cudaEventRecord(ln.ev_front, st));
        CK(cudaEventRecord(ln.ev_handoff, st));
        st = ln.tail;                                  // the rest of the batch runs on the high-priority stream
        CK(cudaStreamWaitEvent(st, ln.ev_handoff, 0));

        BleParams p{};
        p.aa = h->cfg.access_addr;
        p.aa_mask = h->cfg.access_mask ? h->cfg.access_mask : 0xFFFFFFFFu;
        p.crc_init_internal = crc_init_internal(h->cfg.crc_init);
        p.n_out = (int32_t)n_out;
        p.m_origin = (int32_t)pre_out;
        p.n_windows = (int32_t)div_up(body_out, kWindow);
        p.first_window = first_window;
        p.first_capture = first_capture;
        p.n_captures = n_captures;
        p.n_channels = h->n_ble_ch;
        ln.last_p = p; ln.last_lay = lay; ln.last_ble = true;
        BackTotals tot{};
        int r = launch_ble_back(h, ln, p, lay, ln.d_frames, st, &tot);
        if (r != SNRX_OK) return r;
        CK(cudaMemcpyAsync(ln.d_totals + 0, tot.frames, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(ln.d_totals + 1, tot.cands, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    }
    if (h->has_zb && !h->has_ble) {
        CK(cudaEventRecord(ln.ev_handoff, st));        // Zigbee only: front end and chains all on the tail stream
        st = ln.tail;
        CK(cudaStreamWaitEvent(st, ln.ev_handoff, 0));
    }
    if (h->has_zb) {
        const uint32_t first_segment = (uint32_t)(((uint64_t)first_window * kWindow) / h->cfg.zb_segment);
        if (!h->has_ble) CK(cudaEventRecord(ln.ev_front0, st));
        int r = zb_process(ln.zb, h->cfg, x, n_captures, n_samples, x_stride, n_out, pre_out, body_out, first_segment,
                           first_capture, ln.d_frames, h->frame_cap, ln.d_totals, h->has_ble, st, h->sm_count,
                           h->launches, h->err, h->has_ble ? nullptr : ln.ev_front);
        if (r != SNRX_OK) return r;
    }
    if (h->cfg.flags & SNRX_F_RF_METRICS) {        // radio metrics of the final list, from the input the front end read
        RfArgs ra{};
        ra.x = x; ra.stride = x_stride; ra.n_in = (int64_t)n_samples; ra.n_out = (int32_t)n_out;
        ra.nt = h->wideband ? h->pfb_nt : 0;
        ra.origin = (int64_t)first_window * kWindow - (int64_t)pre_out; ra.first_capture = first_capture;
        ra.taps_ble = h->d_taps_flat; ra.taps_zb = h->d_rf_taps_zb; ra.gauss = h->d_rf_gauss;
        ra.frames = ln.d_frames; ra.totals = ln.d_totals; ra.frame_cap = h->frame_cap; ra.out = ln.d_rf;
        k_frame_rf<<<h->sm_count * 2, 32 * kRfWarps, rf_smem_bytes(ra.nt), st>>>(ra);
        h->launches++;
        CK(cudaGetLastError());
    }
    // export: device frame list -> pinned host memory; on this lane's stream, so it overlaps the other lane's front end
    ExportXchg xa{};
    if (h->xchg.connected) {
        for (uint32_t r = 0; r < h->xchg.world; r++) xa.peer[r] = h->xchg.peer[r];
        xa.world = h->xchg.world; xa.rank = h->xchg.rank; xa.cap = h->xchg.cap; xa.slot = (uint32_t)(h->seq_process % SNRX_XCHG_SLOTS);
    }
    k_export_frames<<<32, 256, 0, st>>>(ln.d_frames, ln.d_totals, ln.frames, ln.totals, h->frame_cap, (unsigned long long)h->seq_process, xa);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ln.ev_done, st));
    ln.pending = true; ln.done = false;
    ln.caps = n_captures; ln.n_in = n_samples; ln.n_out = n_out; ln.launches = h->launches;
    h->seq_process++;
    h->b_caps = n_captures; h->b_n_in = n_samples; h->b_n_out = n_out;
    h->batch_valid = true;
    h->last_lane = li;
    return SNRX_OK;
}

// wait for the oldest queued batch, fill its stats; does not consume it
static int finish_oldest(snrx_handle* h, Lane** out_lane) {
    Lane& sl = h->lane[h->seq_poll % kLanes];
    if (!sl.pending) return fail(h, SNRX_ESTATE, "snrx_poll without a queued batch");
    if (!sl.done) {
        CK(cudaSetDevice(h->device));
        CK(cudaEventSynchronize(sl.ev_done));
        const uint32_t n_ble = sl.totals[0], n_cand = sl.totals[1], n_zb = sl.totals[2];
        h->stats.candidates = n_cand;
        sl.done = true;
        sl.n_frames = 0;
        if (n_cand > h->cand_cap) { sl.pending = false; h->seq_poll++; return fail(h, SNRX_EOVERFLOW, "access-address candidates exceed capacity (raise max_frames)"); }
        if ((uint64_t)n_ble + n_zb > h->frame_cap) { sl.pending = false; h->seq_poll++; return fail(h, SNRX_EOVERFLOW, "frames exceed max_frames"); }
        if (sl.totals[3]) { sl.pending = false; h->seq_poll++; return fail(h, SNRX_EOVERFLOW, "a Zigbee chain found more frames than its segment has slots"); }
        sl.n_frames = n_ble + n_zb;
        float ms = 0.f, msf = 0.f;
        cudaEventElapsedTime(&ms, sl.ev_start, sl.ev_done);
        cudaEventElapsedTime(&msf, sl.ev_front0, sl.ev_front);
        const uint32_t ok = sl.totals[5];               // counted by k_export_frames
        h->stats.samples_in = (uint64_t)sl.caps * sl.n_in;
        h->stats.channel_samples = (uint64_t)sl.caps * sl.n_out * (h->n_ble_ch + h->n_zb_ch);
        h->stats.frames = sl.n_frames;
        h->stats.frames_crc_ok = ok;
        h->stats.kernel_launches = (uint32_t)sl.launches;
        h->stats.gpu_ms = ms;
        h->stats.gpu_ms_frontend = msf;
    }
    *out_lane = &sl;
    return SNRX_OK;
}

extern "C" {

int snrx_process(snrx_t* h, const float* iq, uint32_t n_captures, uint64_t n_samples, uint64_t stride_samples,
                 const snrx_shard_t* shard, int is_device_ptr) {
    return process_impl(h, iq, kFmtCf32, n_captures, n_samples, stride_samples, shard, is_device_ptr);
}

int snrx_process_sc8(snrx_t* h, const int8_t* iq, uint32_t n_captures, uint64_t n_samples, uint64_t stride_samples,
                     const snrx_shard_t* shard, int is_device_ptr) {
    return process_impl(h, iq, kFmtSc8, n_captures, n_samples, stride_samples, shard, is_device_ptr);
}

int snrx_debug_process_bits(snrx_t* h, const uint32_t* words, uint32_t n_captures, uint64_t n_samples,
                            const snrx_shard_t* shard) {
    if (!h) return SNRX_EINVAL;
    if (!words) return fail(h, SNRX_EINVAL, "snrx_debug_process_bits: words is NULL");
    if (h->has_zb) return fail(h, SNRX_EINVAL, "snrx_debug_process_bits: BLE-only modes (an 802.15.4 receiver needs its input)");
    if (h->cfg.flags & (SNRX_F_RF_METRICS | SNRX_F_KEEP_STREAMS))
        return fail(h, SNRX_EINVAL, "snrx_debug_process_bits: no input or channel stream to measure or keep");
    return process_impl(h, nullptr, kFmtCf32, n_captures, n_samples, 0, shard, 0, words);
}

int snrx_poll(snrx_t* h, snrx_frame_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    Lane* sl = nullptr;
    int r = finish_oldest(h, &sl);
    if (r != SNRX_OK) return r;
    if (n_out) *n_out = sl->n_frames;
    if (out) {                                   // copying the frames out consumes the batch
        memcpy(out, sl->frames, sizeof(snrx_frame_t) * (size_t)std::min(cap, sl->n_frames));
        sl->pending = false;
        h->polled_lane = (int)(sl - h->lane);
        h->polled_frames_dev = sl->d_frames;
        h->polled_rf_dev = sl->d_rf;
        h->seq_poll++;
    }
    return SNRX_OK;
}

int snrx_poll_view(snrx_t* h, const snrx_frame_t** frames, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    Lane* sl = nullptr;
    int r = finish_oldest(h, &sl);
    if (r != SNRX_OK) return r;
    if (frames) *frames = sl->frames;
    if (n_out) *n_out = sl->n_frames;
    sl->pending = false;
    h->polled_lane = (int)(sl - h->lane);
    h->polled_frames_dev = sl->d_frames;
    h->polled_rf_dev = sl->d_rf;
    h->seq_poll++;
    return SNRX_OK;
}

int snrx_polled_frames_device(snrx_t* h, const snrx_frame_t** frames_dev, uint32_t* n_out) {
    if (!h || h->polled_lane < 0) return SNRX_ESTATE;
    if (frames_dev) *frames_dev = h->polled_frames_dev;
    if (n_out) *n_out = h->lane[h->polled_lane].n_frames;
    return SNRX_OK;
}

int snrx_frame_rf(snrx_t* h, snrx_frame_rf_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (!(h->cfg.flags & SNRX_F_RF_METRICS)) return fail(h, SNRX_ESTATE, "snrx_frame_rf: create the engine with SNRX_F_RF_METRICS");
    if (h->polled_lane < 0) return fail(h, SNRX_ESTATE, "snrx_frame_rf needs a polled batch");
    const uint32_t n = h->lane[h->polled_lane].n_frames;
    if (n_out) *n_out = n;
    if (!out || n == 0) return SNRX_OK;
    if (cap < n) return fail(h, SNRX_ERANGE, "radio-metrics buffer smaller than the batch");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpy(out, h->polled_rf_dev, sizeof(snrx_frame_rf_t) * (size_t)n, cudaMemcpyDeviceToHost));
    return SNRX_OK;
}

int snrx_frames_device(snrx_t* h, void** frames_dev, void** count_dev) {
    if (!h || !h->batch_valid) return SNRX_ESTATE;
    Lane& sl = h->lane[h->last_lane];                                   // lane of the most recent snrx_process
    if (frames_dev) *frames_dev = sl.d_frames;
    if (count_dev) *count_dev = sl.d_totals;
    return SNRX_OK;
}

constexpr uint32_t kDevSlots = 1u << 19;      // open addressing, at most 2^18 senders (load factor 1/2)

static int adv_init(snrx_handle* h) {
    if (h->adv_stream) return SNRX_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMalloc((void**)&h->d_adv, sizeof(snrx_adv_t) * (size_t)h->frame_cap));
    CK(cudaMalloc((void**)&h->d_devtab, sizeof(snrx::DevSlot) * (size_t)kDevSlots));
    CK(cudaMalloc((void**)&h->d_devout, sizeof(snrx_device_t) * (size_t)(kDevSlots / 2)));
    CK(cudaMalloc((void**)&h->d_adv_counters, 4 * sizeof(uint32_t)));
    CK(cudaMemset(h->d_devtab, 0, sizeof(snrx::DevSlot) * (size_t)kDevSlots));
    CK(cudaMemset(h->d_adv_counters, 0, 4 * sizeof(uint32_t)));
    CK(cudaStreamCreateWithFlags(&h->adv_stream, cudaStreamNonBlocking));
    return SNRX_OK;
}

int snrx_ble_adv_summary(snrx_t* h, snrx_adv_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (h->polled_lane < 0) return fail(h, SNRX_ESTATE, "snrx_ble_adv_summary needs a polled batch");
    int r = adv_init(h);
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    const uint32_t n = h->lane[h->polled_lane].n_frames;
    if (n_out) *n_out = n;
    if (n == 0) return SNRX_OK;
    if (out && cap < n) return fail(h, SNRX_ERANGE, "summary buffer smaller than the batch");
    cudaStream_t st = h->adv_stream;
    if (h->dev_count >= kDevSlots / 2) return fail(h, SNRX_EOVERFLOW, "sender table full (2^18 devices)");
    k_ble_adv_summary<<<(n + 255) / 256, 256, 0, st>>>(h->polled_frames_dev, n, h->d_adv, h->d_adv_counters + 0);
    k_ble_adv_devices<<<(n + 255) / 256, 256, 0, st>>>(h->polled_frames_dev, h->d_adv, n, h->d_devtab, kDevSlots - 1, h->d_adv_counters + 1);
    CK(cudaGetLastError());
    uint32_t c[4];
    CK(cudaMemcpyAsync(c, h->d_adv_counters, sizeof c, cudaMemcpyDeviceToHost, st));
    if (out) CK(cudaMemcpyAsync(out, h->d_adv, sizeof(snrx_adv_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    h->dev_count = c[1];
    h->dev_dropped = c[2];
    return SNRX_OK;
}

int snrx_ble_connections(snrx_t* h, snrx_conn_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (h->polled_lane < 0) return fail(h, SNRX_ESTATE, "snrx_ble_connections needs a polled batch");
    int r = adv_init(h);
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    if (!h->d_conn) {
        CK(cudaMalloc((void**)&h->d_conn, sizeof(snrx_conn_t) * (size_t)h->frame_cap));
        CK(cudaMalloc((void**)&h->d_conn_flags, sizeof(uint32_t) * ((size_t)h->frame_cap + 1)));
        CK(cudaMalloc((void**)&h->d_conn_offsets, sizeof(uint32_t) * ((size_t)h->frame_cap + 1)));
        CK(cudaMalloc((void**)&h->d_conn_scratch, sizeof(uint32_t) * scan_scratch_items(h->frame_cap)));
    }
    const uint32_t n = h->lane[h->polled_lane].n_frames;
    if (n_out) *n_out = 0;
    if (n == 0) return SNRX_OK;
    cudaStream_t st = h->adv_stream;
    k_ble_conn_flag<<<(n + 255) / 256, 256, 0, st>>>(h->polled_frames_dev, n, h->d_conn_flags);
    exclusive_scan(h->d_conn_flags, n, h->d_conn_offsets, h->d_conn_scratch, st);
    k_ble_conn_fill<<<(n + 255) / 256, 256, 0, st>>>(h->polled_frames_dev, n, h->d_conn_flags, h->d_conn_offsets, h->d_conn, h->frame_cap);
    CK(cudaGetLastError());
    uint32_t total = 0;
    CK(cudaMemcpyAsync(&total, h->d_conn_offsets + n, sizeof total, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (n_out) *n_out = total;
    if (out && total) {
        if (cap < total) return fail(h, SNRX_ERANGE, "connection buffer smaller than the number of CONNECT_REQs");
        CK(cudaMemcpy(out, h->d_conn, sizeof(snrx_conn_t) * (size_t)total, cudaMemcpyDeviceToHost));
    }
    return SNRX_OK;
}

}  // extern "C"

// The lane of the polled batch, for the calls that search its BLE bit streams again (snrx_ble_follow, snrx_ble_aux,
// snrx_ble_coded, snrx_ble_periodic, snrx_ble_bis): it must hold BLE streams -- of a wideband mode if `wideband` -- that no later batch has overwritten.
static int polled_bits_lane(snrx_handle* h, const char* name, bool wideband, Lane** out) {
    const std::string n = name;
    if (h->polled_lane < 0) return fail(h, SNRX_ESTATE, (n + " needs a polled batch").c_str());
    Lane& ln = h->lane[h->polled_lane];
    if (!h->has_ble || (wideband && !h->wideband) || !ln.last_ble)
        return fail(h, SNRX_ESTATE, (n + (wideband ? ": the polled batch has no wideband BLE bit streams" : ": the polled batch has no BLE bit streams")).c_str());
    if (ln.pending) return fail(h, SNRX_ESTATE, (n + ": the batch's bit streams have been overwritten (call before the second-next snrx_process)").c_str());
    *out = &ln;
    return SNRX_OK;
}

// the polled lane's bit streams as the pointer rounds read them
static AuxGeom aux_geom_of(const Lane& ln) {
    const BleParams& p = ln.last_p;
    AuxGeom g{};
    g.bits = ln.d_bits; g.lay = ln.last_lay; g.n_out = p.n_out;
    g.base = (int64_t)kWindow * p.first_window - p.m_origin;
    g.first_capture = p.first_capture; g.n_captures = p.n_captures;
    return g;
}

// what the pointer rounds of snrx_ble_aux and snrx_ble_coded (and snrx_ble_periodic's scans) share, allocated by the first
// call of any of them
static int round_buffers_init(snrx_handle* h) {
    if (h->d_aux_whiten) return SNRX_OK;
    CK(cudaMalloc((void**)&h->d_round_flags, sizeof(uint32_t) * ((size_t)h->frame_cap + 1)));
    CK(cudaMalloc((void**)&h->d_round_offsets, sizeof(uint32_t) * ((size_t)h->frame_cap + 1)));
    CK(cudaMalloc((void**)&h->d_round_scratch, sizeof(uint32_t) * scan_scratch_items(h->frame_cap)));
    std::vector<uint8_t> wh(40 * SNRX_AUX_MAX_BYTES);
    for (int ch = 0; ch < 40; ch++) make_whiten_bytes(ch, wh.data() + ch * SNRX_AUX_MAX_BYTES, SNRX_AUX_MAX_BYTES);
    CK(cudaMalloc((void**)&h->d_aux_whiten, wh.size()));
    CK(cudaMemcpy(h->d_aux_whiten, wh.data(), wh.size(), cudaMemcpyHostToDevice));
    return SNRX_OK;
}

// The pointer rounds of snrx_ble_aux and snrx_ble_coded, one per depth: the pointers of depth d come from the entries of
// depth d - 1, src are those of the first round.  Appends to `list` from *total on, up to the list kind's maximum depth, and
// leaves the list's length in *total; SNRX_EOVERFLOW with `overflow` if it would pass max_frames.
template <int L>
static int run_pointer_rounds(snrx_handle* h, AuxSrcT<L> src, AuxEntry<L>* list, const AuxGeom& g, cudaStream_t st,
                              uint32_t* total, const char* overflow) {
    const AaTables tabs = make_aa_tables(kAuxAdvAa, 0xFFFFFFFFu);
    const uint32_t crc_init = crc_init_internal(0x555555u);
    uint32_t t = *total;
    while (src.n > 0 && src.depth <= AuxKind<L>::kMaxDepth + 1) {
        k_ble_aux_flag<<<div_up(src.n, 256), 256, 0, st>>>(src, h->d_round_flags);
        exclusive_scan(h->d_round_flags, src.n, h->d_round_offsets, h->d_round_scratch, st);
        uint32_t m = 0;
        CK(cudaMemcpyAsync(&m, h->d_round_offsets + src.n, sizeof m, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (m == 0) break;
        if ((uint64_t)t + m > h->frame_cap) return fail(h, SNRX_EOVERFLOW, overflow);
        k_ble_aux_fill<<<div_up(src.n, 256), 256, 0, st>>>(src, h->d_round_flags, h->d_round_offsets, list, t, g);
        const int gs = grid_for(h, m, 4, 8);
        k_ble_aux_search<L><<<gs, 128, 0, st>>>(list, t, t + m, g, h->d_crc_tab, h->d_aux_whiten, crc_init, tabs);
        if constexpr (AuxKind<L>::kCoded) {
            const CodedTables ct = make_coded_tables();
            k_ble_coded_window<<<gs, 128, 0, st>>>(list, t, t + m, g, ct);
            k_ble_coded_decode<<<grid_for(h, m, kCodedGroups, 8), 8 * kCodedGroups, 0, st>>>(list, t, t + m, g, ct, h->d_crc_tab,
                                                                                              h->d_aux_whiten, crc_init);
        }
        k_ble_aux_first<L><<<grid_for(h, m, 8, 8), 256, 0, st>>>(list, t, t + m);
        CK(cudaGetLastError());
        src.frames = nullptr; src.first = t; src.n = m; src.depth++;
        t += m;
    }
    *total = t;
    return SNRX_OK;
}

// *n_out = total; the list's entries into out (cap entries) if asked for
template <class E>
static int copy_list_out(snrx_handle* h, const char* name, const E* list, uint32_t total, E* out, uint32_t cap, uint32_t* n_out,
                         cudaStream_t st) {
    if (n_out) *n_out = total;
    if (out && total) {
        if (cap < total) return fail(h, SNRX_ERANGE, (std::string(name) + ": buffer smaller than the list").c_str());
        CK(cudaMemcpyAsync(out, list, sizeof(E) * (size_t)total, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return SNRX_OK;
}

// The snrx_ble_periodic list of the polled batch into h->d_sync (*total entries), the aux list it comes from built into
// h->d_aux first with the pointer rounds of snrx_ble_aux; *ln is the polled lane.  Shared by snrx_ble_periodic and
// snrx_ble_bis (`name` in their errors).
static int periodic_list(snrx_handle* h, const char* name, Lane** ln_out, uint32_t* total_out) {
    const std::string nm = name;
    Lane* ln = nullptr;
    int r = polled_bits_lane(h, name, true, &ln);
    if (r != SNRX_OK) return r;
    *ln_out = ln;
    CK(cudaSetDevice(h->device));
    if ((r = round_buffers_init(h)) != SNRX_OK) return r;
    if (!h->d_aux) CK(cudaMalloc((void**)&h->d_aux, sizeof(snrx_ble_aux_t) * (size_t)h->frame_cap));
    if (!h->d_sync) {
        CK(cudaMalloc((void**)&h->d_sync_trains, sizeof(SyncTrain) * (size_t)h->frame_cap));
        CK(cudaMalloc((void**)&h->d_sync, sizeof(snrx_ble_sync_t) * (size_t)h->frame_cap));
    }
    cudaStream_t st = ln->tail;                                  // the lane is idle: its bit streams stay as the batch left them
    const AuxGeom g = aux_geom_of(*ln);
    AuxSrc src{};                                                // the aux list, exactly as snrx_ble_aux builds it
    src.frames = h->polled_frames_dev; src.list = h->d_aux; src.first = 0; src.n = ln->n_frames; src.depth = 0;
    uint32_t n_aux = 0;
    r = run_pointer_rounds(h, src, h->d_aux, g, st, &n_aux, (nm + ": more auxiliary pointers than max_frames").c_str());
    if (r != SNRX_OK) return r;
    uint32_t total = 0;
    if (n_aux) {
        // the trains: flags / offsets over the aux list (n_aux <= max_frames fits the round buffers)
        k_ble_sync_flag<<<grid_for(h, n_aux, 8, 8), 256, 0, st>>>(h->d_aux, n_aux, h->d_round_flags);
        exclusive_scan(h->d_round_flags, n_aux, h->d_round_offsets, h->d_round_scratch, st);
        k_ble_sync_fill<<<div_up(n_aux, 256), 256, 0, st>>>(h->d_aux, n_aux, h->d_round_flags, h->d_round_offsets, h->d_sync_trains);
        uint32_t n_trains = 0;
        CK(cudaMemcpyAsync(&n_trains, h->d_round_offsets + n_aux, sizeof n_trains, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (n_trains) {
            // the events: counts / offsets per train, then one entry per listed event, then the search
            k_ble_sync_count<<<div_up(n_trains, 256), 256, 0, st>>>(h->d_sync_trains, n_trains, g, h->d_round_flags);
            exclusive_scan(h->d_round_flags, n_trains, h->d_round_offsets, h->d_round_scratch, st);
            CK(cudaMemcpyAsync(&total, h->d_round_offsets + n_trains, sizeof total, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (total > h->frame_cap) return fail(h, SNRX_EOVERFLOW, (nm + ": more periodic events than max_frames").c_str());
            if (total) {
                k_ble_sync_events<<<div_up(total, 256), 256, 0, st>>>(h->d_sync_trains, n_trains, h->d_round_offsets, total, g, h->d_sync);
                k_ble_sync_search<<<grid_for(h, total, 4, 8), 128, 0, st>>>(h->d_sync, total, g, h->d_crc_tab, h->d_aux_whiten);
            }
        }
        CK(cudaGetLastError());
    }
    *total_out = total;
    return SNRX_OK;
}

extern "C" {

int snrx_ble_follow(snrx_t* h, uint32_t access_addr, uint32_t crc_init, snrx_frame_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    Lane* ln = nullptr;
    int r = polled_bits_lane(h, "snrx_ble_follow", false, &ln);
    if (r != SNRX_OK) return r;
    if (access_addr == 0u) return fail(h, SNRX_EINVAL, "snrx_ble_follow: access_addr must have a bit set (see snrx_create)");
    CK(cudaSetDevice(h->device));
    if (!h->d_follow) CK(cudaMalloc((void**)&h->d_follow, sizeof(snrx_frame_t) * (size_t)h->frame_cap));
    cudaStream_t st = ln->tail;                                  // the lane is idle: its working set and streams are free
    BleParams p = ln->last_p;
    p.aa = access_addr;
    p.aa_mask = 0xFFFFFFFFu;
    p.crc_init_internal = crc_init_internal(crc_init);
    BackTotals dev{};
    r = launch_ble_back(h, *ln, p, ln->last_lay, h->d_follow, st, &dev);
    if (r != SNRX_OK) return r;
    uint32_t tot[2] = {0, 0};
    CK(cudaMemcpyAsync(&tot[0], dev.frames, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&tot[1], dev.cands, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (tot[1] > h->cand_cap) return fail(h, SNRX_EOVERFLOW, "access-address candidates exceed capacity (raise max_frames)");
    if (tot[0] > h->frame_cap) return fail(h, SNRX_EOVERFLOW, "frames exceed max_frames");
    if (n_out) *n_out = tot[0];
    if (out && tot[0]) {
        if (cap < tot[0]) return fail(h, SNRX_ERANGE, "frame buffer smaller than the number of frames");
        CK(cudaMemcpy(out, h->d_follow, sizeof(snrx_frame_t) * (size_t)tot[0], cudaMemcpyDeviceToHost));
    }
    return SNRX_OK;
}

int snrx_ble_aux(snrx_t* h, snrx_ble_aux_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (n_out) *n_out = 0;
    Lane* ln = nullptr;
    int r = polled_bits_lane(h, "snrx_ble_aux", true, &ln);
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    if ((r = round_buffers_init(h)) != SNRX_OK) return r;
    if (!h->d_aux) CK(cudaMalloc((void**)&h->d_aux, sizeof(snrx_ble_aux_t) * (size_t)h->frame_cap));
    cudaStream_t st = ln->tail;                                  // the lane is idle: its bit streams stay as the batch left them
    AuxSrc src{};                                                // depth 0: the pointers of the polled records
    src.frames = h->polled_frames_dev; src.list = h->d_aux; src.first = 0; src.n = ln->n_frames; src.depth = 0;
    uint32_t total = 0;
    r = run_pointer_rounds(h, src, h->d_aux, aux_geom_of(*ln), st, &total, "snrx_ble_aux: more auxiliary pointers than max_frames");
    if (r != SNRX_OK) return r;
    return copy_list_out(h, "snrx_ble_aux", h->d_aux, total, out, cap, n_out, st);
}

int snrx_ble_coded(snrx_t* h, snrx_ble_coded_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (n_out) *n_out = 0;
    Lane* ln = nullptr;
    int r = polled_bits_lane(h, "snrx_ble_coded", true, &ln);
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    if ((r = round_buffers_init(h)) != SNRX_OK) return r;
    if (!h->d_coded) CK(cudaMalloc((void**)&h->d_coded, sizeof(snrx_ble_coded_t) * (size_t)h->frame_cap));
    const BleParams& p = ln->last_p;
    CodedGeom cg{};
    cg.g = aux_geom_of(*ln);
    cg.body_lo = p.m_origin; cg.body_hi = p.m_origin + p.n_windows * kWindow;
    cg.tiles_per_stream = (uint32_t)div_up(p.n_out, kCodedTile);
    const uint32_t n_tiles = cg.tiles_per_stream * 3u * p.n_captures;
    cudaStream_t st = ln->tail;                                  // the lane is idle: its bit streams stay as the batch left them
    const CodedTables ct = make_coded_tables();
    const uint32_t crc_init = crc_init_internal(0x555555u);
    // the primaries: count per tile, offsets, then the entries in (capture, channel, sample) order, decoded.  The tile scan
    // runs in the lane's access-address scan buffers, which sit idle once the batch is polled: n_tiles + 1 =
    // 3 caps ceil(n_out / 2048) + 1 <= caps 40 ceil(bits_words_for(max_out) / 32) + 1 items of d_counts / d_offsets, and
    // scan_scratch_items is monotonic, so d_scratch is large enough too.
    uint32_t total = 0;
    if (n_tiles) {
        k_ble_coded_scan<false><<<n_tiles, kCodedScanThreads, 0, st>>>(cg, ct, ln->d_counts, nullptr, nullptr);
        exclusive_scan(ln->d_counts, n_tiles, ln->d_offsets, ln->d_scratch, st);
        CK(cudaMemcpyAsync(&total, ln->d_offsets + n_tiles, sizeof total, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (total > h->frame_cap) return fail(h, SNRX_EOVERFLOW, "snrx_ble_coded: more entries than max_frames");
        if (total) {
            k_ble_coded_scan<true><<<n_tiles, kCodedScanThreads, 0, st>>>(cg, ct, ln->d_counts, ln->d_offsets, h->d_coded);
            k_ble_coded_decode<<<grid_for(h, total, kCodedGroups, 8), 8 * kCodedGroups, 0, st>>>(h->d_coded, 0, total, cg.g, ct, h->d_crc_tab,
                                                                                                h->d_aux_whiten, crc_init);
            CK(cudaGetLastError());
        }
    }
    AuxSrcT<kCodedList> src{};                                   // depth 1: the pointers of the primaries
    src.frames = nullptr; src.list = h->d_coded; src.first = 0; src.n = total; src.depth = 1;
    r = run_pointer_rounds(h, src, h->d_coded, cg.g, st, &total, "snrx_ble_coded: more entries than max_frames");
    if (r != SNRX_OK) return r;
    return copy_list_out(h, "snrx_ble_coded", h->d_coded, total, out, cap, n_out, st);
}

int snrx_ble_periodic(snrx_t* h, snrx_ble_sync_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (n_out) *n_out = 0;
    Lane* ln = nullptr;
    uint32_t total = 0;
    const int r = periodic_list(h, "snrx_ble_periodic", &ln, &total);
    if (r != SNRX_OK) return r;
    return copy_list_out(h, "snrx_ble_periodic", h->d_sync, total, out, cap, n_out, ln->tail);
}

int snrx_ble_bis(snrx_t* h, snrx_ble_bis_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (n_out) *n_out = 0;
    Lane* ln = nullptr;
    uint32_t n_sync = 0;
    int r = periodic_list(h, "snrx_ble_bis", &ln, &n_sync);
    if (r != SNRX_OK) return r;
    if (!h->d_bis) {
        CK(cudaMalloc((void**)&h->d_bigs, sizeof(BigGroup) * (size_t)h->frame_cap));
        CK(cudaMalloc((void**)&h->d_bis, sizeof(snrx_ble_bis_t) * (size_t)h->frame_cap));
    }
    cudaStream_t st = ln->tail;                                  // the lane is idle: its bit streams stay as the batch left them
    const AuxGeom g = aux_geom_of(*ln);
    uint32_t total = 0;
    if (n_sync) {
        // the BIGs: flags / offsets over the periodic list (n_sync <= max_frames fits the round buffers)
        k_ble_big_flag<<<grid_for(h, n_sync, 8, 8), 256, 0, st>>>(h->d_sync, n_sync, h->d_round_flags);
        exclusive_scan(h->d_round_flags, n_sync, h->d_round_offsets, h->d_round_scratch, st);
        k_ble_big_fill<<<div_up(n_sync, 256), 256, 0, st>>>(h->d_sync, n_sync, h->d_round_flags, h->d_round_offsets, h->d_bigs);
        uint32_t n_bigs = 0;
        CK(cudaMemcpyAsync(&n_bigs, h->d_round_offsets + n_sync, sizeof n_bigs, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (n_bigs) {
            // the subevents: counts / offsets per BIG, then one entry per subevent of a listed event, then the search
            // The counts are summed on the host in 64 bits before the (32-bit) scan: each is at most max_frames + 1, but
            // n_bigs of them could wrap a 32-bit sum past the overflow test.  Once the sum is at most max_frames the scan
            // cannot wrap.
            k_ble_big_count<<<div_up(n_bigs, 256), 256, 0, st>>>(h->d_bigs, n_bigs, g, h->frame_cap, h->d_round_flags);
            std::vector<uint32_t> counts(n_bigs);
            CK(cudaMemcpyAsync(counts.data(), h->d_round_flags, sizeof(uint32_t) * (size_t)n_bigs, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            uint64_t sum = 0;
            for (uint32_t c : counts) sum += c;
            if (sum > h->frame_cap) return fail(h, SNRX_EOVERFLOW, "snrx_ble_bis: more BIS subevents than max_frames");
            total = (uint32_t)sum;
            exclusive_scan(h->d_round_flags, n_bigs, h->d_round_offsets, h->d_round_scratch, st);
            if (total) {
                k_ble_bis_events<<<div_up(total, 256), 256, 0, st>>>(h->d_bigs, n_bigs, h->d_round_offsets, total, g, h->d_bis);
                k_ble_sync_search<<<grid_for(h, total, 4, 8), 128, 0, st>>>(h->d_bis, total, g, h->d_crc_tab, h->d_aux_whiten);
            }
        }
        CK(cudaGetLastError());
    }
    return copy_list_out(h, "snrx_ble_bis", h->d_bis, total, out, cap, n_out, st);
}

int snrx_zb_mac_summary(snrx_t* h, snrx_zbmac_t* out, uint32_t cap, uint32_t* n_out) {
    if (!h) return SNRX_EINVAL;
    if (h->polled_lane < 0) return fail(h, SNRX_ESTATE, "snrx_zb_mac_summary needs a polled batch");
    int r = adv_init(h);                                       // shares the analytics stream
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    if (!h->d_zbmac) CK(cudaMalloc((void**)&h->d_zbmac, sizeof(snrx_zbmac_t) * (size_t)h->frame_cap));
    const uint32_t n = h->lane[h->polled_lane].n_frames;
    if (n_out) *n_out = n;
    if (n == 0) return SNRX_OK;
    if (out && cap < n) return fail(h, SNRX_ERANGE, "summary buffer smaller than the batch");
    cudaStream_t st = h->adv_stream;
    k_zb_mac_summary<<<(n + 255) / 256, 256, 0, st>>>(h->polled_frames_dev, n, h->d_zbmac);
    CK(cudaGetLastError());
    if (out) CK(cudaMemcpyAsync(out, h->d_zbmac, sizeof(snrx_zbmac_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SNRX_OK;
}

int snrx_ble_devices(snrx_t* h, snrx_device_t* out, uint32_t cap, uint32_t* n_out, int reset) {
    if (!h) return SNRX_EINVAL;
    int r = adv_init(h);
    if (r != SNRX_OK) return r;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->adv_stream;
    // one batch can add up to frame_cap senders, so the counter may run past what the export buffer holds: the table is
    // then over its design load and the surplus senders are reported as an overflow, never read out of bounds
    const bool over = h->dev_count > kDevSlots / 2;
    const uint32_t n = over ? kDevSlots / 2 : h->dev_count;
    if (n_out) *n_out = n;
    if (out && n) {
        if (cap < n) return fail(h, SNRX_ERANGE, "device buffer smaller than the table");
        CK(cudaMemsetAsync(h->d_adv_counters + 3, 0, sizeof(uint32_t), st));
        k_ble_adv_export<<<(kDevSlots + 255) / 256, 256, 0, st>>>(h->d_devtab, kDevSlots, h->d_devout, kDevSlots / 2, h->d_adv_counters + 3);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out, h->d_devout, sizeof(snrx_device_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    const bool dropped = h->dev_dropped != 0 || over;
    if (reset) {
        CK(cudaMemsetAsync(h->d_devtab, 0, sizeof(snrx::DevSlot) * (size_t)kDevSlots, st));
        CK(cudaMemsetAsync(h->d_adv_counters, 0, 4 * sizeof(uint32_t), st));
        CK(cudaStreamSynchronize(st));
        h->dev_count = h->dev_dropped = 0;
    }
    if (dropped) return fail(h, SNRX_EOVERFLOW, "more than 2^18 distinct senders: some were not recorded");
    return SNRX_OK;
}

// ---- frame exchange between the engines of a node ----------------------------------------------------------------------
static size_t xchg_slot_bytes(const snrx_handle* h) { return ((size_t)h->xchg.cap + 1) * sizeof(snrx_frame_t); }

int snrx_exchange_create(snrx_t* h, uint32_t rank, uint32_t world, uint32_t cap_records, void* handle_out) {
    if (!h || !handle_out) return SNRX_EINVAL;
    if (world < 1 || world > SNRX_XCHG_MAX_WORLD || rank >= world || cap_records == 0) return fail(h, SNRX_EINVAL, "exchange: rank / world / capacity out of range");
    if (h->xchg.d_recv) return fail(h, SNRX_ESTATE, "exchange already created");
    static_assert(sizeof(cudaIpcMemHandle_t) == SNRX_XCHG_HANDLE_BYTES, "CUDA IPC handle size");
    CK(cudaSetDevice(h->device));
    h->xchg.rank = rank; h->xchg.world = world; h->xchg.cap = cap_records;
    const size_t bytes = (size_t)world * SNRX_XCHG_SLOTS * xchg_slot_bytes(h);
    CK(cudaMalloc((void**)&h->xchg.d_recv, bytes));
    CK(cudaMemset(h->xchg.d_recv, 0xFF, bytes));                         // batch numbers of all ones: nothing has arrived
    CK(cudaHostAlloc((void**)&h->xchg.h_hdr, sizeof(uint64_t) * 2 * SNRX_XCHG_MAX_WORLD, cudaHostAllocDefault));
    CK(cudaStreamCreateWithFlags(&h->xchg.stream, cudaStreamNonBlocking));
    cudaIpcMemHandle_t ipc;
    CK(cudaIpcGetMemHandle(&ipc, h->xchg.d_recv));
    memcpy(handle_out, &ipc, sizeof ipc);
    CK(cudaDeviceSynchronize());
    return SNRX_OK;
}

int snrx_exchange_connect(snrx_t* h, const void* handles) {
    if (!h || !handles) return SNRX_EINVAL;
    if (!h->xchg.d_recv) return fail(h, SNRX_ESTATE, "snrx_exchange_create first");
    if (h->xchg.connected) return fail(h, SNRX_ESTATE, "exchange already connected");
    CK(cudaSetDevice(h->device));
    for (auto& ln : h->lane) { CK(cudaStreamSynchronize(ln.stream)); CK(cudaStreamSynchronize(ln.tail)); }
    for (uint32_t r = 0; r < h->xchg.world; r++) {
        if (r == h->xchg.rank) { h->xchg.peer[r] = h->xchg.d_recv; continue; }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const unsigned char*)handles + (size_t)r * SNRX_XCHG_HANDLE_BYTES, sizeof ipc);
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
        h->xchg.peer[r] = (unsigned char*)p;
    }
    h->xchg.connected = true;
    return SNRX_OK;
}

int snrx_allgather(snrx_t* h, uint64_t batch_no, snrx_frame_t* out, uint32_t cap, uint32_t* counts, uint32_t* n_out,
                   uint32_t timeout_ms) {
    if (!h) return SNRX_EINVAL;
    if (!h->xchg.connected) return fail(h, SNRX_ESTATE, "snrx_allgather: the engines are not connected (snrx_exchange_connect)");
    CK(cudaSetDevice(h->device));
    const uint32_t world = h->xchg.world, slot = (uint32_t)(batch_no % SNRX_XCHG_SLOTS);
    const size_t sb = xchg_slot_bytes(h);
    const unsigned char* base = h->xchg.d_recv + (size_t)slot * sb;          // slot of rank 0; ranks are SLOTS * sb apart
    const auto t0 = std::chrono::steady_clock::now();
    for (;;) {
        // the headers of all ranks in one strided copy
        CK(cudaMemcpy2DAsync(h->xchg.h_hdr, 16, base, SNRX_XCHG_SLOTS * sb, 16, world, cudaMemcpyDeviceToHost, h->xchg.stream));
        CK(cudaStreamSynchronize(h->xchg.stream));
        bool all = true;
        for (uint32_t r = 0; r < world; r++) all = all && h->xchg.h_hdr[2 * r + 1] == batch_no;
        if (all) break;
        const auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        if ((uint64_t)ms >= timeout_ms) return fail(h, SNRX_ESTATE, "snrx_allgather: batch did not arrive from every rank in time");
        std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
    uint64_t total = 0; bool over = false;
    for (uint32_t r = 0; r < world; r++) {
        const uint64_t c = h->xchg.h_hdr[2 * r];
        if (counts) counts[r] = (uint32_t)c;
        over = over || c > h->xchg.cap;
        total += c;
    }
    if (n_out) *n_out = (uint32_t)total;
    if (over) return fail(h, SNRX_EOVERFLOW, "snrx_allgather: a rank had more records than the exchange capacity");
    if (out) {
        if (total > cap) return fail(h, SNRX_ERANGE, "snrx_allgather: output buffer too small");
        size_t off = 0;
        for (uint32_t r = 0; r < world; r++) {
            const size_t c = (size_t)h->xchg.h_hdr[2 * r];
            if (c) CK(cudaMemcpyAsync(out + off, base + (size_t)r * SNRX_XCHG_SLOTS * sb + sizeof(snrx_frame_t), c * sizeof(snrx_frame_t),
                                      cudaMemcpyDeviceToHost, h->xchg.stream));
            off += c;
        }
        CK(cudaStreamSynchronize(h->xchg.stream));
        // only the pieces a record uses travelled: what lies behind its payload is whatever the slot held before
        for (size_t i = 0; i < off; i++)
            if (out[i].len < sizeof out[i].bytes) memset(out[i].bytes + out[i].len, 0, sizeof out[i].bytes - out[i].len);
    }
    return SNRX_OK;
}

// ---- N4: synthetic captures on the GPU ---------------------------------------------------------------------------------
int snrx_synth_wideband(int device, const snrx_tx_burst_t* bursts, uint32_t n_bursts, const uint8_t* data, uint64_t n_data,
                        const int32_t* bins, uint32_t n_bins, const float* taps, const double* gauss, uint64_t n_steps,
                        float sigma, uint64_t seed, float* iq_out, int out_is_device) {
    snrx_handle* h = nullptr;
    if (!bins || !taps || !gauss || !iq_out || n_bins == 0 || n_bins > (uint32_t)kTxMaxBins || n_steps == 0) return fail(nullptr, SNRX_EINVAL, "synth: bad argument");
    if (n_bursts && (!bursts || !data)) return fail(nullptr, SNRX_EINVAL, "synth: bursts without data");
    CK(cudaSetDevice(device));
    // bursts in start order, so that every time chunk only launches the bursts that reach into it
    std::vector<snrx_tx_burst_t> sorted(bursts, bursts + n_bursts);
    std::stable_sort(sorted.begin(), sorted.end(), [](const snrx_tx_burst_t& a, const snrx_tx_burst_t& b) { return a.start < b.start; });
    int64_t longest = 0;
    for (const auto& b : sorted) {
        if (b.bin_slot >= n_bins || (uint64_t)b.data_offset + (b.proto == SNRX_PROTO_BLE ? (b.n_units + 7) / 8 : b.n_units) > n_data)
            return fail(nullptr, SNRX_EINVAL, "synth: burst outside its data / bins");
        longest = std::max<int64_t>(longest, tx_burst_samples(b));
    }
    const int64_t hist = kTxTapsPerPhase - 1;
    const int64_t chunk = std::min<int64_t>((int64_t)n_steps, 1 << 20);
    const int64_t slen = chunk + hist;
    snrx_tx_burst_t* d_bursts = nullptr; uint8_t* d_data = nullptr; float2* d_streams = nullptr; float* d_taps = nullptr;
    double* d_gauss = nullptr; float2* d_out = nullptr;
    cudaStream_t st = nullptr;
    auto cleanup = [&]() {
        for (void* p : {(void*)d_bursts, (void*)d_data, (void*)d_streams, (void*)d_taps, (void*)d_gauss}) if (p) cudaFree(p);
        if (d_out && !out_is_device) cudaFree(d_out);
        if (st) cudaStreamDestroy(st);
    };
#define SCK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { g_err = std::string(#call) + " -> " + cudaGetErrorString(e__); cleanup(); return e__ == cudaErrorMemoryAllocation ? SNRX_ENOMEM : SNRX_ECUDA; } } while (0)
    SCK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    SCK(cudaFuncSetAttribute(k_tx_synthesis, cudaFuncAttributeMaxDynamicSharedMemorySize, kTxSynSmem));
    if (n_bursts) {
        SCK(cudaMalloc((void**)&d_bursts, sizeof(snrx_tx_burst_t) * n_bursts));
        SCK(cudaMemcpyAsync(d_bursts, sorted.data(), sizeof(snrx_tx_burst_t) * n_bursts, cudaMemcpyHostToDevice, st));
        SCK(cudaMalloc((void**)&d_data, n_data));
        SCK(cudaMemcpyAsync(d_data, data, n_data, cudaMemcpyHostToDevice, st));
    }
    SCK(cudaMalloc((void**)&d_streams, sizeof(float2) * (size_t)n_bins * (size_t)slen));
    SCK(cudaMalloc((void**)&d_taps, sizeof(float) * kTxTapsPerPhase * 24));
    SCK(cudaMemcpyAsync(d_taps, taps, sizeof(float) * kTxTapsPerPhase * 24, cudaMemcpyHostToDevice, st));
    SCK(cudaMalloc((void**)&d_gauss, sizeof(double) * 16));
    SCK(cudaMemcpyAsync(d_gauss, gauss, sizeof(double) * 16, cudaMemcpyHostToDevice, st));
    if (out_is_device) d_out = reinterpret_cast<float2*>(iq_out);
    else SCK(cudaMalloc((void**)&d_out, sizeof(float2) * 24 * (size_t)chunk));
    size_t first = 0;                                            // bursts before `first` end before the current chunk
    for (int64_t p0 = 0; p0 < (int64_t)n_steps; p0 += chunk) {
        const int64_t steps = std::min<int64_t>(chunk, (int64_t)n_steps - p0);
        const int64_t c0 = p0 - hist, c1 = p0 + steps;           // channel-rate samples [c0, c1) live in the streams
        SCK(cudaMemsetAsync(d_streams, 0, sizeof(float2) * (size_t)n_bins * (size_t)slen, st));
        while (first < sorted.size() && sorted[first].start + longest <= c0) first++;
        size_t last = first;
        while (last < sorted.size() && sorted[last].start < c1) last++;
        if (last > first) {
            TxModArgs m{};
            m.bursts = d_bursts + first; m.n_bursts = (uint32_t)(last - first); m.data = d_data; m.streams = d_streams;
            m.stream_len = slen; m.chunk_start = c0; m.gauss = d_gauss;
            k_tx_modulate<<<(unsigned)(last - first), 256, 0, st>>>(m);
        }
        TxSynArgs sa{};
        sa.streams = d_streams; sa.stream_len = slen; sa.n_bins = (int32_t)n_bins;
        for (uint32_t k = 0; k < n_bins; k++) sa.bins[k] = ((bins[k] % 96) + 96) % 96;
        sa.g = d_taps; sa.n_steps = steps; sa.sample0 = p0 * 24; sa.sigma = sigma; sa.seed = seed;
        sa.out = out_is_device ? d_out + (size_t)p0 * 24 : d_out;
        k_tx_synthesis<<<(unsigned)((steps + kTxTileP - 1) / kTxTileP), 256, kTxSynSmem, st>>>(sa);
        SCK(cudaGetLastError());
        if (!out_is_device) {
            SCK(cudaMemcpyAsync(iq_out + (size_t)p0 * 24 * 2, d_out, sizeof(float2) * 24 * (size_t)steps, cudaMemcpyDeviceToHost, st));
            SCK(cudaStreamSynchronize(st));
        }
    }
    SCK(cudaStreamSynchronize(st));
#undef SCK
    cleanup();
    return SNRX_OK;
}

int snrx_stats(snrx_t* h, snrx_stats_t* s) {
    if (!h || !s) return SNRX_EINVAL;
    *s = h->stats;
    return SNRX_OK;
}

int snrx_debug_stage(snrx_t* h, int stage, void* out, uint64_t cap_bytes, uint64_t* n_bytes) {
    if (!h || !h->batch_valid) return SNRX_ESTATE;
    CK(cudaSetDevice(h->device));
    Lane& ln = h->lane[h->last_lane];                                    // streams of the most recent snrx_process
    CK(cudaStreamSynchronize(ln.stream));
    CK(cudaStreamSynchronize(ln.tail));
    const void* src = nullptr;
    uint64_t bytes = 0;
    switch (stage) {
        case SNRX_STAGE_BLE_Q8:
            if (!ln.d_q8) return fail(h, SNRX_ESTATE, "create the engine with SNRX_F_KEEP_STREAMS");
            src = ln.d_q8; bytes = (uint64_t)h->b_caps * h->n_ble_ch * h->b_n_out * 2; break;
        case SNRX_STAGE_CHAN_CF32:
            if (h->cfg.mode == SNRX_MODE_ZB_WB16) {
                int r = zb_debug_stage(ln.zb, stage, h->b_caps, h->b_n_out, &src, &bytes);
                if (r != SNRX_OK) return fail(h, r, "create the engine with SNRX_F_KEEP_STREAMS");
                break;
            }
            if (!ln.d_cf) return fail(h, SNRX_ESTATE, "create a wideband engine with SNRX_F_KEEP_STREAMS");
            src = ln.d_cf; bytes = (uint64_t)h->b_caps * h->n_ble_ch * h->b_n_out * 8; break;
        case SNRX_STAGE_BLE_BITS: {
            if (!ln.d_bits) return SNRX_ESTATE;
            src = ln.d_bits; bytes = (uint64_t)h->b_caps * h->n_ble_ch * bits_words_for(h->b_n_out) * 4; break;
        }
        default: {
            int r = zb_debug_stage(ln.zb, stage, h->b_caps, h->b_n_out, &src, &bytes);
            if (r != SNRX_OK) return fail(h, r, "stage not available in this mode");
        }
    }
    if (n_bytes) *n_bytes = bytes;
    if (out) {
        if (cap_bytes < bytes) return fail(h, SNRX_ERANGE, "debug buffer too small");
        CK(cudaMemcpy(out, src, bytes, cudaMemcpyDeviceToHost));
    }
    return SNRX_OK;
}

int snrx_host_alloc(void** p, uint64_t bytes) {
    if (!p) return SNRX_EINVAL;
    return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? SNRX_OK : SNRX_ENOMEM;
}
int snrx_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? SNRX_OK : SNRX_ECUDA; }

}  // extern "C"
