// synth.cuh -- SURVEY 8(f) row N4: the transmit side on the GPU -- GFSK and O-QPSK modulators and the x24 synthesis
// filterbank that lifts per-channel 4 Msps bursts into one 96 Msps capture, with AWGN.
//
// Reference statements of the waveforms: vendor/BTLE/host/btle-tools/src/btle_tx.c:1111-1149 (gen_sample_from_phy_bit,
// float version: NRZ impulses every SAMPLE_PER_SYMBOL samples convolved with the Gaussian taps, phase = running sum times
// pi * MOD_IDX / SAMPLE_PER_SYMBOL, sample = cos / sin of it; constants :103-128) and
// snout/grc-blocks/transmitter_OQPSK.py:96-111 (nibble -> 16 complex chip pairs, each repeated 4 times and multiplied by the
// half-sine [0, sin(pi/4), 1, sin(3pi/4)], Q delayed by 2 samples) with the SHR / PHR of
// scapy-radio/gnuradio/gr-zigbee/lib/preamble_prefixer_scapy_impl.cc:48-52,67-88.  snout_b200/synth.py states the same in
// numpy (it is what the tests compare these kernels with); the frame SCHEDULE (which bytes, where, which carrier offset)
// is drawn on the host by synth.py and handed over as snrx_tx_burst_t records, so both sides place the same frames.
//
//   k_tx_modulate   one CTA per burst: bits / chips -> complex baseband at 4 Msps, times amp * exp(j(phase0 + 2 pi cfo n / fs)),
//                   added into the stream of the burst's filterbank bin (bursts of two protocols may share a bin);
//   k_tx_synthesis  x[24 p + rho] = sum_i g[24 i + rho] * A[p - i][(24 p + rho) mod 96],  A[q][r] = sum_k s_k[q] W^(bin_k r):
//                   a CTA computes the 96-point transform rows it needs into shared memory, then the polyphase
//                   interpolation, adds white Gaussian noise from a counter-based generator (Philox-4x32-10 + Box-Muller,
//                   a function of (seed, sample index) only) and writes cf32.
#pragma once
#include "common.cuh"

namespace snrx {

constexpr int kTxTapsPerPhase = 16;                 // synthesis prototype: 24 * 16 taps
constexpr int kTxTileP = 32;                        // channel-rate steps per CTA of k_tx_synthesis
constexpr int kTxRows = kTxTileP + kTxTapsPerPhase - 1;
constexpr int kTxMaxBins = 48;
constexpr int kTxSynSmem = 8 * (kTxMaxBins * kTxRows + kTxRows * 97 + 96) + 4 * kTxTapsPerPhase * 24;

// 32-chip PN sequence of data symbol s (IEEE 802.15.4 2450 MHz O-QPSK PHY), chip k in bit k
SNRX_HD uint32_t tx_zb_chips(int s) {
    // symbol 0: 1101 1001 1100 0011 0101 0010 0010 1110 (chip 0 first)
    const uint32_t pn0 = 0x744AC39Bu;               // chip k = bit k
    const int k = 4 * (s & 7);
    uint32_t c = k ? ((pn0 << k) | (pn0 >> (32 - k))) : pn0;      // cyclic shift right by k chips: c[j] = pn0[j - k]
    if (s & 8) c ^= 0xAAAAAAAAu;                    // odd chips inverted
    return c;
}

// GFSK instantaneous frequency at sample i: freq[i] = sum_j gauss[i - 4 j] (2 bit_j - 1) over the bits whose impulse lies
// under the 16 taps; the phase is (pi h / 4) sum_{m < i} freq[m], h = 0.5.  bit(j) returns bit j of the burst (0 / 1).
constexpr double kGfskPhasePerFreq = 3.14159265358979323846 * 0.5 / 4.0;
template <class Bit>
SNRX_HD double gfsk_freq(const double* gauss, int64_t i, int64_t n_bits, Bit bit) {
    double fr = 0.0;
    for (int t = 0; t < 4; t++) {
        const int64_t j = (i >> 2) - t;
        const int tap = (int)(i - 4 * j);
        if (j >= 0 && j < n_bits && tap < 16) fr += gauss[tap] * (bit(j) ? 1.0 : -1.0);
    }
    return fr;
}

#if defined(__CUDACC__)
struct TxModArgs {
    const snrx_tx_burst_t* bursts; uint32_t n_bursts;
    const uint8_t* data;            // packed burst data: BLE phy bits LSB first (8 per byte), 802.15.4 PPDU bytes
    float2* streams;                // [n_bins][stream_len] baseband at 4 Msps (zeroed by the caller)
    int64_t stream_len;             // channel-rate samples per stream (this chunk)
    int64_t chunk_start;            // channel-rate index of the chunk's first sample in the capture
    const double* gauss;            // [16] Gaussian taps of the GFSK modulator
};

// burst length in channel-rate samples
__host__ __device__ inline int64_t tx_burst_samples(const snrx_tx_burst_t& b) {
    return b.proto == SNRX_PROTO_BLE ? (int64_t)b.n_units * 4 + 15 : (int64_t)b.n_units * 2 * 64 + 2;   // impulses every 4 samples convolved with 16 taps / bytes * 2 symbols * 64 + Q delay
}

__global__ void __launch_bounds__(256) k_tx_modulate(TxModArgs a) {
    __shared__ double scan[256];
    __shared__ double carry;
    const snrx_tx_burst_t b = a.bursts[blockIdx.x];
    const int64_t n = tx_burst_samples(b);
    const int64_t lo = b.start - a.chunk_start;                      // position inside this chunk (may be negative / beyond)
    if (lo + n <= 0 || lo >= a.stream_len) return;
    const uint8_t* d = a.data + b.data_offset;
    float2* out = a.streams + (size_t)b.bin_slot * a.stream_len;
    const double two_pi = 6.283185307179586476925286766559;
    const double dphi = two_pi * (double)b.cfo_hz / 4.0e6;
    if (threadIdx.x == 0) carry = 0.0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        double re = 0.0, im = 0.0, fr = 0.0;
        if (b.proto == SNRX_PROTO_BLE) {
            if (i < n) fr = gfsk_freq(a.gauss, i, (int64_t)b.n_units, [&](int64_t j) { return (d[j >> 3] >> (j & 7)) & 1; });
            // exclusive prefix sum of fr over the burst (block scan, carry between rounds)
            scan[threadIdx.x] = fr;
            __syncthreads();
            for (int o = 1; o < (int)blockDim.x; o <<= 1) {
                const double v = threadIdx.x >= (unsigned)o ? scan[threadIdx.x - o] : 0.0;
                __syncthreads();
                scan[threadIdx.x] += v;
                __syncthreads();
            }
            const double incl = scan[threadIdx.x] + carry;
            const double ph = (incl - fr) * kGfskPhasePerFreq;
            __syncthreads();
            if (threadIdx.x == blockDim.x - 1) carry = incl;
            __syncthreads();
            double s, c;
            sincos(ph, &s, &c);
            re = c; im = s;
        } else if (i < n) {
            // chips of symbol sym = nibble (low first) of PPDU byte; I takes the even chips, Q the odd ones, 2 samples later
            const double hs[4] = {0.0, 0.70710678118654752440, 1.0, 0.70710678118654752440};
            auto chip = [&](int64_t c) -> double {                   // chip c of the burst, +-1
                const int64_t sym = c >> 5;
                const int nib = (d[sym >> 1] >> (4 * (sym & 1))) & 15;
                return ((tx_zb_chips(nib) >> (c & 31)) & 1u) ? 1.0 : -1.0;
            };
            const int64_t n_pairs = (int64_t)b.n_units * 2 * 16;     // chip pairs = samples / 4
            if ((i >> 2) < n_pairs) re = chip(2 * (i >> 2)) * hs[i & 3];
            const int64_t m = i - 2;
            if (m >= 0 && (m >> 2) < n_pairs) im = chip(2 * (m >> 2) + 1) * hs[m & 3];
        }
        if (i < n) {
            double s, c;
            sincos((double)b.phase0 + dphi * (double)i, &s, &c);
            const double xr = (double)b.amp * (re * c - im * s), xi = (double)b.amp * (re * s + im * c);
            const int64_t p = lo + i;
            if (p >= 0 && p < a.stream_len) {
                atomicAdd(&out[p].x, (float)xr);
                atomicAdd(&out[p].y, (float)xi);
            }
        }
    }
}

// ---- counter-based noise: Philox-4x32-10 keyed by the seed, counter = sample index; 4 uniforms -> 2 normal pairs
__device__ __forceinline__ uint4 tx_philox(uint64_t ctr, uint64_t key) {
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0x5EED5EEDu, c3 = 0u;
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float2 tx_normal_pair(uint32_t u0, uint32_t u1) {      // Box-Muller
    const float r = sqrtf(-2.0f * __logf(((float)u0 + 1.0f) * 2.3283064365386963e-10f));
    float s, c;
    __sincosf((float)u1 * (6.2831853071795864769f * 2.3283064365386963e-10f), &s, &c);
    return make_float2(r * c, r * s);
}

struct TxSynArgs {
    const float2* streams;          // [n_bins][stream_len]; stream index q = channel-rate step of this chunk + kTxTapsPerPhase - 1 (history in front)
    int64_t stream_len;
    int32_t n_bins;
    int32_t bins[kTxMaxBins];       // filterbank bin (0..95) of every stream
    const float* g;                 // [16][24] synthesis taps, g[i][rho] = g[24 i + rho] (gain 24)
    float2* out;                    // [n_steps * 24] cf32 at 96 Msps
    int64_t n_steps;                // channel-rate steps to produce
    int64_t sample0;                // input-rate index of out[0] in the capture (noise counter, rotation phase)
    float sigma;                    // noise standard deviation per component
    uint64_t seed;
};

__global__ void __launch_bounds__(256) k_tx_synthesis(TxSynArgs a) {
    extern __shared__ __align__(16) unsigned char tx_smem[];
    float2 (*S)[kTxRows] = reinterpret_cast<float2 (*)[kTxRows]>(tx_smem);                                   // s_k[q] of the tile (18 KB)
    float2 (*A)[96 + 1] = reinterpret_cast<float2 (*)[96 + 1]>(tx_smem + sizeof(float2) * kTxMaxBins * kTxRows);   // A[q][r] (36.5 KB)
    float2* W = reinterpret_cast<float2*>(tx_smem + sizeof(float2) * (kTxMaxBins * kTxRows + kTxRows * 97));
    float* G = reinterpret_cast<float*>(W + 96);
    const int tid = threadIdx.x;
    const int64_t p0 = (int64_t)blockIdx.x * kTxTileP;               // first step of the tile
    for (int i = tid; i < 96; i += blockDim.x) { float s, c; sincospif(2.0f * (float)i / 96.0f, &s, &c); W[i] = make_float2(c, s); }
    for (int i = tid; i < kTxTapsPerPhase * 24; i += blockDim.x) G[i] = a.g[i];
    for (int i = tid; i < a.n_bins * kTxRows; i += blockDim.x) {
        const int k = i / kTxRows, q = i - k * kTxRows;              // row q = step p0 - 15 + q = stream index p0 + q
        const int64_t si = p0 + q;
        S[k][q] = si < a.stream_len ? a.streams[(size_t)k * a.stream_len + si] : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // the rotation exp(j 2 pi bin n / 96) is a function of n mod 96 of the CAPTURE index: r below is relative to the tile's
    // first output sample 24 p0 + sample0, whose residue is added
    const int r0 = (int)(((p0 * 24 + a.sample0) % 96 + 96) % 96);
    for (int e = tid; e < kTxRows * 96; e += blockDim.x) {
        const int q = e / 96, r = e - q * 96;
        const int rr = (r + r0) % 96;
        float ar = 0.f, ai = 0.f;
        for (int k = 0; k < a.n_bins; k++) {
            const float2 w = W[(a.bins[k] * rr) % 96];
            const float2 s = S[k][q];
            ar = fmaf(s.x, w.x, fmaf(-s.y, w.y, ar));
            ai = fmaf(s.x, w.y, fmaf(s.y, w.x, ai));
        }
        A[q][r] = make_float2(ar, ai);
    }
    __syncthreads();
    const float amp = a.sigma;
    for (int o = tid; o < kTxTileP * 24 / 2; o += blockDim.x) {      // two consecutive outputs per iteration (one Philox call)
        float2 res[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int n = 2 * o + h, p = n / 24, rho = n - 24 * p;   // output 24 (p0 + p) + rho
            float xr = 0.f, xi = 0.f;
#pragma unroll
            for (int i = 0; i < kTxTapsPerPhase; i++) {
                const float2 v = A[p + (kTxTapsPerPhase - 1) - i][(24 * p + rho) % 96];
                const float gg = G[i * 24 + rho];
                xr = fmaf(gg, v.x, xr); xi = fmaf(gg, v.y, xi);
            }
            res[h] = make_float2(xr, xi);
        }
        const int64_t gidx = (p0 * 24 + 2 * (int64_t)o);            // index inside this launch's output
        if (amp > 0.f) {
            const uint4 u = tx_philox((uint64_t)(a.sample0 + gidx) >> 1, a.seed);
            const float2 n0 = tx_normal_pair(u.x, u.y), n1 = tx_normal_pair(u.z, u.w);
            res[0].x += amp * n0.x; res[0].y += amp * n0.y; res[1].x += amp * n1.x; res[1].y += amp * n1.y;
        }
        if (gidx + 1 < a.n_steps * 24) *reinterpret_cast<float4*>(a.out + gidx) = make_float4(res[0].x, res[0].y, res[1].x, res[1].y);
        else if (gidx < a.n_steps * 24) a.out[gidx] = res[0];
    }
}
#endif

}  // namespace snrx
