// ble_coded.cuh -- BLE Long Range: ADV_EXT_INDs on the LE Coded PHY on channels 37..39, found in the slicer bit streams the
// batch left in HBM by their FEC-coded access address, Viterbi-decoded, and followed down their AuxPtrs on every PHY.  The
// contract is stated in include/snoutrx.h above snrx_ble_coded_t; oracle/coded_oracle.py restates it.
//
// Launched by snrx_ble_coded:
//   k_ble_coded_scan<false> / exclusive_scan / k_ble_coded_scan<true>   d(n) at every position of the three primary streams,
//                                                                       the local minima <= T counted per tile, then written
//                                                                       in (capture, channel, sample) order
//   k_ble_coded_decode                                                  8 lanes (one trellis state each) per packet: CI, the
//                                                                       header and full Viterbi runs, de-whitening, CRC
//   then one round per chain depth: k_ble_aux_flag / _fill / _search / _first (ble_aux.cuh, on snrx_ble_coded_t) with
//   k_ble_coded_window + k_ble_coded_decode for the Coded targets
#pragma once
#include "ble_aux.cuh"
#include "common.cuh"
#include "scan.cuh"

namespace snrx {

static_assert(sizeof(snrx_ble_coded_t) == 320 && sizeof(snrx_ble_coded_t) % 16 == 0, "snrx_ble_coded_t layout (include/snoutrx.h, _abi.CODED_DTYPE)");
static_assert(offsetof(snrx_ble_coded_t, bytes) == 52, "snrx_ble_coded_t layout");

constexpr int kCodedCiSamples = 160;           // CI + TERM1: 10 coded bits at 16 decisions
constexpr int kCodedBlock2 = kCodedAaSamples + kCodedCiSamples;
constexpr int kCodedHalf = 16;                 // the local-minimum neighbourhood on each side
constexpr uint32_t kCodedT = SNRX_CODED_T;
constexpr uint32_t kCodedInf = 1u << 20;       // path metric of an unreached state
constexpr int kCodedMaxSteps = 8 * 255 + 43;   // info bits of the longest block 2
constexpr uint8_t kCodedDecode = 0xFD;         // internal: found, to be decoded by k_ble_coded_decode
constexpr int kCodedTile = 2048;               // scan positions per block: 8 per thread
constexpr int kCodedScanThreads = 256;
constexpr int kCodedScanWords = (kCodedTile + 2 * kCodedHalf + kCodedAaSamples + 32) / 32 + 2;
constexpr int kCodedGroups = 8;                // packets per block of k_ble_coded_decode (8 lanes each)

// The sample-level patterns, LSB first: aa[k] bit i = P[32 k + i]; ci[v][w] bit i = sample 32 w + i of CI value v's
// pattern (v coded from the state after the AA, then TERM1).
struct CodedTables {
    uint32_t aa[32];
    uint32_t ci[4][5];
};

// 16 samples of one S=8 coded bit x: symbols x x !x !x, 4 samples each
SNRX_HD constexpr uint32_t coded_s8_pattern(int x) { return x ? 0x00FFu : 0xFF00u; }

// rate 1/2, K = 4: D1 | D2 << 1 | D3 << 2, a0 = u^D1^D2^D3, a1 = u^D2^D3
inline int coded_encode(const int* u, int n, int state, int* out) {
    for (int i = 0; i < n; i++) {
        const int d1 = state & 1, d2 = (state >> 1) & 1, d3 = (state >> 2) & 1;
        out[2 * i] = u[i] ^ d1 ^ d2 ^ d3;
        out[2 * i + 1] = u[i] ^ d2 ^ d3;
        state = ((state << 1) | u[i]) & 7;
    }
    return state;
}

inline CodedTables make_coded_tables() {
    CodedTables t{};
    int u[32], c[64];
    for (int i = 0; i < 32; i++) u[i] = (int)((kAuxAdvAa >> i) & 1u);
    const int st = coded_encode(u, 32, 0, c);
    for (int k = 0; k < 32; k++) t.aa[k] = coded_s8_pattern(c[2 * k]) | (coded_s8_pattern(c[2 * k + 1]) << 16);
    for (int v = 0; v < 4; v++) {
        const int ub[5] = {v & 1, v >> 1, 0, 0, 0};
        int cc[10];
        coded_encode(ub, 5, st, cc);
        for (int w = 0; w < 5; w++) t.ci[v][w] = coded_s8_pattern(cc[2 * w]) | (coded_s8_pattern(cc[2 * w + 1]) << 16);
    }
    return t;
}

struct CodedGeom {                // the polled batch, as AuxGeom, plus the body of a shard and the scan's tiling
    AuxGeom g;
    int32_t body_lo, body_hi;     // local samples whose primaries belong to this batch
    uint32_t tiles_per_stream;
};

#if defined(__CUDACC__)
// 32 decisions from local sample m (stream_words = the stream's word 0, lead words included)
__device__ __forceinline__ uint32_t coded_read32(const uint32_t* __restrict__ stream_words, int m) {
    const int x = m + 32 * kBitsLeadWords, w = x >> 5;
    return funnel_r(__ldg(stream_words + w), __ldg(stream_words + w + 1), x & 31);
}

// d(n) clamped to T + 1 (exact for every use: a position above T can neither be a packet nor beat one); n + 1023 usable
__device__ __forceinline__ uint32_t coded_distance(const uint32_t* __restrict__ stream_words, int n, const CodedTables& t) {
    uint32_t acc = 0;
#pragma unroll 8
    for (int k = 0; k < 32; k++) {
        acc += __popc(coded_read32(stream_words, n + 32 * k) ^ t.aa[k]);
        if ((k & 7) == 7 && acc > kCodedT) return kCodedT + 1;
    }
    return acc;
}

__device__ __forceinline__ void coded_zero(snrx_ble_coded_t& r) {
    uint4* d = reinterpret_cast<uint4*>(&r);
#pragma unroll
    for (int q = 0; q < (int)(sizeof(snrx_ble_coded_t) / 16); q++) d[q] = make_uint4(0u, 0u, 0u, 0u);
}

// One block per tile of kCodedTile positions of one (capture, channel 37..39) stream.  d(n) of the tile and 16 positions on
// either side from the stream's words in shared memory; each thread then owns 8 consecutive positions and keeps the strict
// local minima <= T inside the body.  FILL = false: the tile's count; FILL = true: the entries at list[offsets[tile] ...].
template <bool FILL>
__global__ void __launch_bounds__(kCodedScanThreads) k_ble_coded_scan(CodedGeom cg, const __grid_constant__ CodedTables t,
                                                                      uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets,
                                                                      snrx_ble_coded_t* __restrict__ list) {
    __shared__ uint32_t w_s[kCodedScanWords];
    __shared__ uint16_t d_s[kCodedTile + 2 * kCodedHalf];
    const AuxGeom& g = cg.g;
    const uint32_t tile = blockIdx.x, stream = tile / cg.tiles_per_stream, ti = tile % cg.tiles_per_stream;
    const uint32_t cap = stream / 3, ch = 37 + stream % 3;
    const int p0 = (int)ti * kCodedTile;
    const int s0 = p0 - 32;                                       // sample of bit 0 of w_s[0]
    const uint32_t* pw = g.bits + g.lay.index(cap, ch, 0);
    const int nw = (int)g.lay.words_per_stream;
    for (int i = threadIdx.x; i < kCodedScanWords; i += blockDim.x) {
        const int w = kBitsLeadWords + (s0 >> 5) + i;
        w_s[i] = w < nw ? pw[w] : 0u;
    }
    __syncthreads();
    const int last = g.n_out - 2;
    for (int q = threadIdx.x; q < kCodedTile + 2 * kCodedHalf; q += blockDim.x) {
        const int n = p0 - kCodedHalf + q;
        uint32_t d = kCodedT + 1;
        if (n >= 0 && n + kCodedAaSamples - 1 <= last) {
            const int o = q + kCodedHalf, k0 = o >> 5, sh = o & 31;
            uint32_t acc = 0;
#pragma unroll 8
            for (int k = 0; k < 32; k++) {
                acc += __popc(funnel_r(w_s[k0 + k], w_s[k0 + k + 1], sh) ^ t.aa[k]);
                if ((k & 7) == 7 && acc > kCodedT) break;
            }
            d = min(acc, kCodedT + 1);
        }
        d_s[q] = (uint16_t)d;
    }
    __syncthreads();
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int q = kCodedHalf + 8 * threadIdx.x + i, n = p0 + 8 * threadIdx.x + i;
        const uint32_t dn = d_s[q];
        if (dn > kCodedT || n < cg.body_lo || n >= cg.body_hi) continue;
        bool ok = true;
#pragma unroll
        for (int m = 1; m <= kCodedHalf; m++) ok = ok && d_s[q - m] > dn && d_s[q + m] >= dn;
        if (ok) mask |= 1u << i;
    }
    uint32_t total;
    uint32_t k = block_exclusive_scan(__popc(mask), &total);
    if (!FILL) {
        if (threadIdx.x == 0) counts[tile] = total;
        return;
    }
    k += offsets[tile];
    for (; mask; mask &= mask - 1, k++) {
        const int i = __ffs(mask) - 1, n = p0 + 8 * threadIdx.x + i;
        snrx_ble_coded_t& r = list[k];
        coded_zero(r);
        const int64_t si = g.base + n;
        r.sample_index = si; r.win_lo = si; r.win_hi = si;
        r.capture_id = g.first_capture + cap;
        r.parent = 0xFFFFFFFFu;
        r.first = k;
        r.channel = (uint8_t)ch;
        r.phy = SNRX_AUX_PHY_CODED;
        r.phase = (uint8_t)(si & 3);
        r.aa_errors = d_s[kCodedHalf + 8 * threadIdx.x + i];
        r.ci = 0xFF;
        r.status = kCodedDecode;
    }
}

// One warp per Coded target of [i0, i1): the n of its window with the smallest d(n) <= T, the earliest on ties.
__global__ void __launch_bounds__(128) k_ble_coded_window(snrx_ble_coded_t* __restrict__ list, uint32_t i0, uint32_t i1, AuxGeom g,
                                                          const __grid_constant__ CodedTables t) {
    const int lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t k = i0 + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < i1; k += warps) {
        snrx_ble_coded_t& r = list[k];
        if (r.status != kCodedPending) continue;                  // warp-uniform
        const int lo = (int)(r.win_lo - g.base), hi = (int)(r.win_hi - g.base);   // inside the buffer (k_ble_aux_fill)
        const uint32_t* pw = g.bits + g.lay.index(r.capture_id - g.first_capture, r.channel, 0);
        uint64_t best = ~0ull;                                    // d << 32 | n: the smallest d, then the smallest n
        for (int n = lo + lane; n <= hi; n += 32) {
            const uint32_t d = coded_distance(pw, n, t);
            if (d <= kCodedT) best = min(best, ((uint64_t)d << 32) | (uint32_t)n);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
        if (lane == 0) {
            if (best == ~0ull) r.status = SNRX_AUX_NOT_FOUND;
            else {
                const int n = (int)(uint32_t)best;
                const int64_t si = g.base + n;
                r.sample_index = si;
                r.phase = (uint8_t)(si & 3);
                r.aa_errors = (uint16_t)(best >> 32);
                r.status = kCodedDecode;
            }
        }
    }
}

// Eight lanes per entry of [i0, i1) found and not yet decoded, lane s holding trellis state s: the CI choice, then the ACS
// steps (survivors one byte per step in shared memory), the header run's traceback at step 40, the full run to step N and
// its traceback from state 0, by the group's lane 0.
__global__ void __launch_bounds__(8 * kCodedGroups) k_ble_coded_decode(snrx_ble_coded_t* __restrict__ list, uint32_t i0, uint32_t i1,
                                                                            AuxGeom g, const __grid_constant__ CodedTables t,
                                                                            const uint32_t* __restrict__ crc_tab,
                                                                            const uint8_t* __restrict__ whiten /*[40][260]*/,
                                                                            uint32_t crc_init_internal) {
    __shared__ uint32_t crc_s[256];
    __shared__ uint8_t surv_s[kCodedGroups][kCodedMaxSteps + 1];
    __shared__ uint8_t buf_s[kCodedGroups][SNRX_AUX_MAX_BYTES];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_s[i] = crc_tab[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, s = lane & 7, grp = threadIdx.x >> 3;
    const unsigned gm = 0xFFu << (lane & 24);
    uint8_t* surv = surv_s[grp];
    uint8_t* buf = buf_s[grp];
    const uint32_t groups = gridDim.x * (blockDim.x >> 3);
    // predecessors of state s: p0 = s >> 1 (D3 = 0) and p1 = p0 | 4; the coded bits of the transition p -> s (input s & 1)
    const int u = s & 1, p0 = s >> 1, p1 = p0 | 4;
    const int a0_0 = u ^ (__popc(p0) & 1), a1_0 = u ^ (__popc(p0 >> 1) & 1);
    const int a0_1 = u ^ (__popc(p1) & 1), a1_1 = u ^ (__popc(p1 >> 1) & 1);
    for (uint32_t k = i0 + blockIdx.x * (blockDim.x >> 3) + grp; k < i1; k += groups) {
        snrx_ble_coded_t& r = list[k];
        if (r.status != kCodedDecode) continue;                   // uniform in the group
        const int n = (int)(r.sample_index - g.base), last = g.n_out - 2;
        const uint32_t* pw = g.bits + g.lay.index(r.capture_id - g.first_capture, r.channel, 0);
        const uint8_t* wh = whiten + r.channel * SNRX_AUX_MAX_BYTES;
        uint8_t status = SNRX_AUX_TRUNCATED, ci = 0xFF, ok = 0;
        uint32_t metric = 0;
        int nb = 0;
        if (n + kCodedBlock2 - 1 <= last) {
            uint32_t best = ~0u;
            for (int v = 0; v < 4; v++) {
                uint32_t dv = 0;
                for (int w = 0; w < 5; w++) dv += __popc(coded_read32(pw, n + kCodedAaSamples + 32 * w) ^ t.ci[v][w]);
                if (dv < best) { best = dv; ci = (uint8_t)v; }
            }
            if (ci >= 2) status = SNRX_AUX_RESERVED_CI;
            else {
                const bool s8 = ci == 0;
                const int L = s8 ? 16 : 4, start = n + kCodedBlock2;
                uint32_t pm = s == 0 ? 0u : kCodedInf;
                auto acs = [&](int t0, int t1) {
                    for (int st = t0; st < t1; st++) {
                        uint32_t bA0, bB0;
                        if (s8) {
                            const uint32_t x = coded_read32(pw, start + 32 * st);
                            bA0 = __popc((x & 0xFFFFu) ^ coded_s8_pattern(0)); bB0 = __popc((x >> 16) ^ coded_s8_pattern(0));
                        } else {
                            const uint32_t x = coded_read32(pw, start + 8 * st);
                            bA0 = __popc(x & 0xFu); bB0 = __popc((x >> 4) & 0xFu);
                        }
                        const uint32_t bA1 = L - bA0, bB1 = L - bB0;
                        const uint32_t q0 = __shfl_sync(gm, pm, p0, 8), q1 = __shfl_sync(gm, pm, p1, 8);
                        const uint32_t m0 = q0 + (a0_0 ? bA1 : bA0) + (a1_0 ? bB1 : bB0);
                        const uint32_t m1 = q1 + (a0_1 ? bA1 : bA0) + (a1_1 ? bB1 : bB0);
                        const bool take = m1 < m0;
                        pm = take ? m1 : m0;
                        const uint32_t b = __ballot_sync(gm, take);
                        if (s == 0) surv[st] = (uint8_t)(b >> (lane & 24));
                    }
                };
                auto trace = [&](int steps, int state, int nbits) {     // lane s == 0 only: info bits 0..nbits-1 into buf
                    for (int j = 0; j < (nbits + 7) / 8; j++) buf[j] = 0;
                    for (int st = steps - 1; st >= 0; st--) {
                        if (st < nbits) buf[st >> 3] |= (uint8_t)((state & 1) << (st & 7));
                        state = (state >> 1) | (((surv[st] >> state) & 1) << 2);
                    }
                };
                if (start + 80 * L - 1 <= last) {
                    acs(0, 40);
                    uint32_t key = (pm << 3) | (uint32_t)s;             // the lowest metric, then the lowest state
#pragma unroll
                    for (int o = 4; o; o >>= 1) key = min(key, __shfl_xor_sync(gm, key, o, 8));
                    int len = 0;
                    if (s == 0) { trace(40, (int)(key & 7u), 16); len = (buf[1] ^ wh[1]) & 0xFF; }
                    len = __shfl_sync(gm, len, 0, 8);
                    const int N = 8 * len + 43;
                    if (start + 2 * N * L - 1 <= last) {
                        acs(40, N);
                        metric = __shfl_sync(gm, pm, 0, 8);
                        nb = len + 5;
                        status = SNRX_AUX_OK;
                        if (s == 0) {
                            trace(N, 0, 8 * nb);
                            uint32_t crc = crc_init_internal;
                            for (int j = 0; j < nb; j++) {
                                buf[j] ^= wh[j];
                                if (j < nb - 3) crc = (crc_s[(crc ^ buf[j]) & 0xFFu] ^ (crc >> 8)) & 0xFFFFFFu;
                            }
                            const uint32_t recv = (uint32_t)buf[nb - 3] | ((uint32_t)buf[nb - 2] << 8) | ((uint32_t)buf[nb - 1] << 16);
                            ok = crc == recv;
                        }
                    }
                }
            }
        }
        __syncwarp(gm);
        for (int j = s; j < nb; j += 8) r.bytes[j] = buf[j];
        if (s == 0) {
            r.status = status; r.ci = ci; r.len = (uint16_t)nb; r.crc_ok = ok; r.metric = metric;
        }
        __syncwarp(gm);                                           // buf and surv are reused by the group's next entry
    }
}
#endif  // __CUDACC__

}  // namespace snrx
