// ble_aux.cuh -- BLE 5 extended advertising: follow the AuxPtr of every ADV_EXT_IND of a batch (and of the AUX_ADV_IND /
// AUX_CHAIN_IND it finds) to the auxiliary packet on its data channel, on the 1M and 2M PHYs, in the slicer bit streams the
// batch left in HBM.  The contract (pointer sources, window, search, decode, statuses, order) is stated in include/snoutrx.h
// above snrx_ble_aux_t; oracle/aux_oracle.py restates it.
//
// One round per chain depth, launched by snrx_ble_aux (and, templated on the entry type, by snrx_ble_coded: ble_coded.cuh):
//   k_ble_aux_flag / exclusive_scan / k_ble_aux_fill   the pointers of the round, in source order, with their windows and the
//                                                       statuses that need no search
//   k_ble_aux_search                                    one warp per pointer: windowed access-address search, then the decode
//   k_ble_aux_first                                     one warp per entry: the earliest entry that found the same packet
#pragma once
#include "ble_back.cuh"
#include "common.cuh"

namespace snrx {

static_assert(sizeof(snrx_ble_aux_t) == 304 && sizeof(snrx_ble_aux_t) % 16 == 0, "snrx_ble_aux_t layout (include/snoutrx.h, _abi.AUX_DTYPE)");

constexpr uint32_t kAuxAdvAa = 0x8E89BED6u;
constexpr int kAuxGuard = 8;                   // samples on both sides of the window
constexpr uint8_t kAuxPending = 0xFF;          // internal: to be searched

struct AuxPtr {
    int channel, ca, units_us, offset, phy;
};

// pdu = header(2) | payload as stored in the records; n_payload = payload bytes.  True if this is a PDU of type 7 whose extended
// header carries an AuxPtr (with every field in front of it inside the header).
SNRX_HD bool aux_ptr_parse(const uint8_t* pdu, int n_payload, AuxPtr& a) {
    if ((pdu[0] & 0x0F) != 7 || n_payload < 2) return false;
    const uint8_t* p = pdu + 2;
    const int hlen = p[0] & 0x3F;
    if (hlen < 1 || 1 + hlen > n_payload) return false;
    const int flags = p[1];
    if (!(flags & 0x10)) return false;
    const int off = 2 + ((flags & 1) ? 6 : 0) + ((flags & 2) ? 6 : 0) + ((flags & 4) ? 1 : 0) + ((flags & 8) ? 2 : 0);
    if (off + 3 > 1 + hlen) return false;
    const int a0 = p[off], a1 = p[off + 1], a2 = p[off + 2];
    a.channel = a0 & 0x3F;
    a.ca = (a0 >> 6) & 1;
    a.units_us = (a0 & 0x80) ? 300 : 30;
    a.offset = a1 | ((a2 & 0x1F) << 8);
    a.phy = a2 >> 5;
    return true;
}

// [lo, hi] of AA bit 0 positions, relative to the source's AA bit 0 (integer arithmetic only: kernel and oracle agree exactly)
SNRX_HD void aux_window(const AuxPtr& a, int64_t& lo, int64_t& hi) {
    const int64_t U = a.units_us, O = (int64_t)a.offset * U, ppm = a.ca ? 50 : 500;
    lo = (4 * O * (1000000 - ppm)) / 1000000 - kAuxGuard;
    hi = (4 * (O + U) * (1000000 + ppm) + 999999) / 1000000 + kAuxGuard;
}

// Bit-parallel correlation at a symbol stride of 2 samples (2M PHY): bit i of the result is set when the decisions at
// samples i + 2p (p = 0..31) of the word w[0] equal the access address.  w[1], w[2] are the words that follow.
template <class KEEP>
SNRX_HD uint32_t aa_word_hits2(const uint32_t (&w)[3], const AaTables& t, KEEP keep_going) {
    uint32_t m = 0xFFFFFFFFu;
#pragma unroll
    for (int p = 0; p < 32; p++) {
        const int sh = (2 * p) & 31, k = (2 * p) >> 5;
        const uint32_t s = sh ? funnel_r(w[k], w[k + 1], sh) : w[k];
        m &= (s ^ t.want0[p]) | t.dont_care[p];
        if ((p & 3) == 3 && p >= 11 && p < 31) { if (!keep_going(m)) return 0u; }
    }
    return m;
}

// every 2nd bit of x starting at bit 0 (16 bits) -> low 8 bits
SNRX_HD uint32_t compress2(uint32_t x) {
    x &= 0x5555u;
    x = (x | (x >> 1)) & 0x3333u;
    x = (x | (x >> 2)) & 0x0F0Fu;
    x = (x | (x >> 4)) & 0x00FFu;
    return x;
}

// byte j of a packet whose AA bit 0 is at local sample n (decisions b[n + (32 + 8 j + i) sps], i = 0..7, LSB first)
SNRX_HD uint32_t aux_read_byte(const uint32_t* stream_words, int n, int j, int sps) {
    const int m = n + (32 + 8 * j) * sps + 32 * kBitsLeadWords, w = m >> 5, sh = m & 31;
    const uint32_t v = funnel_r(stream_words[w], stream_words[w + 1], sh);
    return sps == 4 ? compress4(v) : compress2(v);
}

struct AuxGeom {                  // the polled batch
    const uint32_t* bits;
    BitsLayout lay;
    int64_t base;                 // capture index of local sample 0 = first_window * 8192 - m_origin
    int32_t n_out;                // channel samples per capture in the buffer
    uint32_t first_capture, n_captures;
};

// What the two lists that share the pointer rounds differ in.  snrx_ble_aux: AUX_ADV_IND = depth 0, 1M / 2M only, AA bit 0
// 32 samples after the preamble on both PHYs.  snrx_ble_coded: primaries = depth 0, Coded targets too, preamble 320 samples
// on Coded (the window is shifted by P(target) - P(source)).
constexpr int kAuxList = 0, kCodedList = 1;
template <int L> struct AuxKind;
template <> struct AuxKind<kAuxList> {
    using Entry = snrx_ble_aux_t;
    static constexpr bool kCoded = false;
    static constexpr uint32_t kMaxDepth = SNRX_AUX_MAX_DEPTH;
    static constexpr int kMaxPhy = SNRX_AUX_PHY_2M;
};
template <> struct AuxKind<kCodedList> {
    using Entry = snrx_ble_coded_t;
    static constexpr bool kCoded = true;
    static constexpr uint32_t kMaxDepth = SNRX_CODED_MAX_DEPTH;
    static constexpr int kMaxPhy = SNRX_AUX_PHY_CODED;
};
template <int L> using AuxEntry = typename AuxKind<L>::Entry;
template <int L>
struct AuxSrcT {                  // where the pointers of one round come from
    const snrx_frame_t* frames;   // snrx_ble_aux at depth 0: the polled records [0, n); else nullptr
    const AuxEntry<L>* list;      // otherwise: the entries [first, first + n) of the previous round
    uint32_t first, n, depth;     // depth of the pointers the round creates
};
using AuxSrc = AuxSrcT<kAuxList>;

SNRX_HD constexpr int aux_preamble(int phy) { return phy == SNRX_AUX_PHY_CODED ? 320 : 32; }
constexpr uint8_t kCodedPending = 0xFE;        // internal: a Coded target, to be searched by k_ble_coded_window
constexpr int kCodedAaSamples = 1024;          // the coded access address: 256 symbols of 4 samples

#if defined(__CUDACC__)
template <int L>
__device__ __forceinline__ bool aux_source(const AuxSrcT<L>& s, uint32_t i, AuxPtr& a, int64_t& at, uint32_t& cap_id, int& phy) {
    phy = SNRX_AUX_PHY_1M;
    if (s.frames) {
        const snrx_frame_t& f = s.frames[i];
        if (f.proto != SNRX_PROTO_BLE || !f.crc_ok || f.channel < 37 || f.channel > 39 || f.access_addr != kAuxAdvAa || f.len < 5)
            return false;
        at = f.sample_index; cap_id = f.capture_id;
        return aux_ptr_parse(f.bytes, (int)f.len - 5, a);
    }
    const uint32_t k = s.first + i;
    const AuxEntry<L>& r = s.list[k];
    if (r.status != SNRX_AUX_OK || !r.crc_ok || r.first != k || r.len < 5) return false;
    at = r.sample_index; cap_id = r.capture_id; phy = r.phy;
    return aux_ptr_parse(r.bytes, (int)r.len - 5, a);
}

template <int L>
__global__ void __launch_bounds__(256) k_ble_aux_flag(AuxSrcT<L> s, uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s.n) return;
    AuxPtr a; int64_t at; uint32_t cap_id; int phy;
    flags[i] = aux_source(s, i, a, at, cap_id, phy) ? 1u : 0u;
}

// the round's entries at list[k0 + offsets[i]]: windows, pre-search statuses, zero bytes
template <int L>
__global__ void __launch_bounds__(256) k_ble_aux_fill(AuxSrcT<L> s, const uint32_t* __restrict__ flags, const uint32_t* __restrict__ offsets,
                                                      AuxEntry<L>* __restrict__ list, uint32_t k0, AuxGeom g) {
    using K = AuxKind<L>;
    using E = AuxEntry<L>;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s.n || !flags[i]) return;
    AuxPtr a; int64_t at; uint32_t cap_id; int src_phy;
    aux_source(s, i, a, at, cap_id, src_phy);
    const uint32_t k = k0 + offsets[i];
    E& r = list[k];
    uint4* d = reinterpret_cast<uint4*>(&r);
#pragma unroll
    for (int q = 0; q < (int)(sizeof(E) / 16); q++) d[q] = make_uint4(0u, 0u, 0u, 0u);
    int64_t lo, hi;
    aux_window(a, lo, hi);
    if constexpr (K::kCoded) {
        at += aux_preamble(a.phy) - aux_preamble(src_phy);
        r.ci = 0xFF;
    }
    r.sample_index = -1;
    r.win_lo = at + lo; r.win_hi = at + hi;
    r.capture_id = cap_id;
    r.parent = s.frames ? i : s.first + i;
    r.first = k;
    r.depth = (uint8_t)s.depth;
    r.channel = (uint8_t)a.channel;
    r.phy = (uint8_t)a.phy;
    uint8_t st = kAuxPending;
    if (s.depth > K::kMaxDepth) st = SNRX_AUX_DEPTH_LIMIT;
    else if (a.channel > 36) st = SNRX_AUX_BAD_CHANNEL;
    else if (a.phy > K::kMaxPhy) st = SNRX_AUX_UNSUPPORTED_PHY;
    else {
        const int sps = a.phy == SNRX_AUX_PHY_2M ? 2 : 4;
        const int span = (K::kCoded && a.phy == SNRX_AUX_PHY_CODED) ? kCodedAaSamples - 1 : 31 * sps;
        const int64_t l = r.win_lo - g.base, e = r.win_hi - g.base + span;        // local first / last decision of the search
        if (l < 0 || e + 1 >= g.n_out) st = SNRX_AUX_OUTSIDE;
        else if (K::kCoded && a.phy == SNRX_AUX_PHY_CODED) st = kCodedPending;
    }
    r.status = st;
}

// The earliest n in [lo, hi] (local samples, inside the buffer) whose 32 decisions at stride sps equal the address of
// `tabs`, or -1: one warp, 32 words per pass.  Shared by snrx_ble_aux and snrx_ble_periodic.
__device__ __forceinline__ int aux_find(const uint32_t* pw, uint32_t nw, int lo, int hi, int sps, const AaTables& tabs, int lane) {
    for (int wb = kBitsLeadWords + (lo >> 5); wb <= kBitsLeadWords + (hi >> 5); wb += 32) {
        const int w = wb + lane;
        const int s0 = 32 * (w - kBitsLeadWords);                 // sample of bit 0 of word w
        uint32_t h;
        auto keep = [](uint32_t m) { return __any_sync(0xffffffffu, m != 0u) != 0; };
        if (sps == 4) {
            uint32_t ww[5];
#pragma unroll
            for (int d = 0; d < 5; d++) ww[d] = ((uint32_t)(w + d) < nw) ? __ldg(pw + w + d) : 0u;
            h = aa_word_hits(ww, tabs, keep);
        } else {
            uint32_t ww[3];
#pragma unroll
            for (int d = 0; d < 3; d++) ww[d] = ((uint32_t)(w + d) < nw) ? __ldg(pw + w + d) : 0u;
            h = aa_word_hits2(ww, tabs, keep);
        }
        // keep start positions lo..hi
        if (s0 + 31 < lo || s0 > hi) h = 0u;
        else {
            if (s0 < lo) h &= 0xFFFFFFFFu << (lo - s0);
            if (s0 + 31 > hi) h &= 0xFFFFFFFFu >> (s0 + 31 - hi);
        }
        const uint32_t any = __ballot_sync(0xffffffffu, h != 0u);
        if (any) {
            const int src = __ffs(any) - 1;
            return __shfl_sync(0xffffffffu, s0 + __ffs(h) - 1, src);
        }
    }
    return -1;
}

// One warp: the packet whose AA bit 0 is at local sample n (found by aux_find) read, de-whitened by `channel` and checked
// with the CRC seeded by crc_init_internal, into the entry's sample_index / phase / len / crc_ok / status / bytes.  buf is
// the warp's SNRX_AUX_MAX_BYTES of shared memory, crc_s the CRC table in shared memory.
template <class E>
__device__ __forceinline__ void aux_decode(E& r, const uint32_t* pw, int n, int sps, int channel, const AuxGeom& g,
                                           const uint32_t* crc_s, const uint8_t* __restrict__ whiten, uint32_t crc_init_internal,
                                           uint8_t* buf, int lane) {
    const int last_usable = g.n_out - 2;
    uint8_t status = SNRX_AUX_TRUNCATED;
    int nb = 0;
    if (n + 47 * sps <= last_usable) {                            // the header's last decision
        const int len = (int)((aux_read_byte(pw, n, 1, sps) ^ whiten[channel * SNRX_AUX_MAX_BYTES + 1]) & 0xFFu);
        if (n + (32 + 8 * (len + 5) - 1) * sps <= last_usable) { nb = len + 5; status = SNRX_AUX_OK; }
    }
    for (int j = lane; j < nb; j += 32) buf[j] = (uint8_t)(aux_read_byte(pw, n, j, sps) ^ whiten[channel * SNRX_AUX_MAX_BYTES + j]);
    __syncwarp();
    for (int j = lane; j < nb; j += 32) r.bytes[j] = buf[j];
    if (lane == 0) {
        uint32_t ok = 0;
        if (nb) {
            uint32_t crc = crc_init_internal;
            for (int j = 0; j < nb - 3; j++) crc = (crc_s[(crc ^ buf[j]) & 0xFFu] ^ (crc >> 8)) & 0xFFFFFFu;
            const uint32_t recv = (uint32_t)buf[nb - 3] | ((uint32_t)buf[nb - 2] << 8) | ((uint32_t)buf[nb - 1] << 16);
            ok = crc == recv;
        }
        const int64_t si = g.base + n;
        r.sample_index = si;
        r.phase = (uint8_t)(si % sps);
        r.len = (uint16_t)nb;
        r.crc_ok = (uint8_t)ok;
        r.status = status;
    }
    __syncwarp();                                                 // buf is reused by the warp's next entry
}

// One warp per entry of [i0, i1) still pending: the earliest full access-address match in the window, then the decode.
template <int L>
__global__ void __launch_bounds__(128) k_ble_aux_search(AuxEntry<L>* __restrict__ list, uint32_t i0, uint32_t i1, AuxGeom g,
                                                        const uint32_t* __restrict__ crc_tab, const uint8_t* __restrict__ whiten /*[40][260]*/,
                                                        uint32_t crc_init_internal, const __grid_constant__ AaTables tabs) {
    __shared__ uint32_t crc_s[256];
    __shared__ uint8_t buf_s[4][SNRX_AUX_MAX_BYTES];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_s[i] = crc_tab[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t k = i0 + blockIdx.x * (blockDim.x >> 5) + wib; k < i1; k += warps) {
        AuxEntry<L>& r = list[k];
        if (r.status != kAuxPending) continue;                    // warp-uniform
        const int sps = r.phy == SNRX_AUX_PHY_2M ? 2 : 4;
        const int lo = (int)(r.win_lo - g.base), hi = (int)(r.win_hi - g.base);   // inside the buffer (k_ble_aux_fill)
        const uint32_t* pw = g.bits + g.lay.index(r.capture_id - g.first_capture, r.channel, 0);
        const int n = aux_find(pw, g.lay.words_per_stream, lo, hi, sps, tabs, lane);
        if (n < 0) { if (lane == 0) r.status = SNRX_AUX_NOT_FOUND; continue; }
        aux_decode(r, pw, n, sps, r.channel, g, crc_s, whiten, crc_init_internal, buf_s[wib], lane);
    }
}

template <class E>
__device__ __forceinline__ bool aux_found(const E& r) { return r.status == SNRX_AUX_OK || r.status == SNRX_AUX_TRUNCATED; }

// One warp per entry of [i0, i1): first = the smallest list index that found the same (capture, channel, AA bit 0, PHY).
template <int L>
__global__ void __launch_bounds__(256) k_ble_aux_first(AuxEntry<L>* __restrict__ list, uint32_t i0, uint32_t i1) {
    using E = AuxEntry<L>;
    const int lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t k = i0 + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < i1; k += warps) {
        const E& r = list[k];
        if (!aux_found(r)) continue;
        uint32_t first = k;
        for (uint32_t b = 0; b < k; b += 32) {
            const uint32_t j = b + lane;
            bool same = false;
            if (j < k) {
                const E& o = list[j];
                same = aux_found(o) && o.sample_index == r.sample_index && o.channel == r.channel && o.capture_id == r.capture_id && o.phy == r.phy;
            }
            const uint32_t m = __ballot_sync(0xffffffffu, same);
            if (m) { first = b + (uint32_t)(__ffs(m) - 1); break; }
        }
        if (lane == 0) list[k].first = first;
    }
}
#endif  // __CUDACC__

}  // namespace snrx
