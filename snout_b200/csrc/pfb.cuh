// pfb.cuh -- wideband polyphase-filterbank channelizer fused with the BLE slicer.
//
// No reference counterpart: Snout retunes one 4 Msps channel at a time
// (snout/util/btle.py:62, snout/core/radio.py:415).  Definition (DESIGN.md "Channelizer",
// restated on the CPU in oracle/pfb_oracle.c):
//
//   y_k[m] = (-j)^(k m) * sum_{n<L} h[n] exp(+j 2 pi k n / 96) x[24 m - n]      M = 96 bins, D = 24
//
// BLE mode needs the 40 even bins only, so the bank is evaluated as a 48-branch bank:
//   v_r[m]   = sum_{p<L/48} h[r + 48 p] x[24 m - r - 48 p]            r = 0..47   (FIR, FP32 FMA)
//   y_2q[m]  = (-1)^(q m) * sum_r v_r[m] exp(+j 2 pi q r / 48)                     (48-point inverse DFT)
// followed, per channel, by the int8-grid quantiser and the reference's one-sample
// cross-product slicer (btle_rx.c:1357-1361); only ONE BIT per channel sample leaves the SM.
//
// One WARP (= one CTA) computes 32 channel-rate samples x 40 channels end to end and emits the 31 slicer
// bits per channel whose successor sample it holds; tiles advance by 31 samples, so they are independent:
// no carry, no stitch pass, no CTA-wide barrier.
//   phase 0  cp.async stages the input tile into shared memory (coalesced 16-byte copies); the tile
//            is laid out flat with a 64-byte skew every 192 samples so that phase 1 is bank-conflict free;
//   phase 1  three passes gi = 0..2, each: FIR of branches r = gi + 3 rl (+24) -- lane (rl, chunk) owns the
//            decimated sequence X_rho[c] = x[24 c - rho], rho = gi + 3 rl, and 8 consecutive output times; the
//            taps of that rho live in registers and each loaded sample feeds up to 16 FMAs (register sliding
//            window) -- then a 4 KB transpose through shared memory (16-byte stores/loads, XOR swizzle) and,
//            one lane per output time, the 16-point inverse DFT over the branches r = gi (mod 3), in
//            registers.  Keeping only one third of the branch outputs in shared memory at a time is what
//            lets 16 warps share an SM.  Pass gi reads its branches in the rotated order of the prime-factor
//            map (fft.cuh Pfa48), so that the 48-point transform needs no twiddles;
//   phase 2  twiddle-free radix-3 combination of the three 16-point transforms (fft.cuh Pfa48), bin rotation,
//            quantisation of the 40 bins that carry a channel, packing of each quantised (I, Q) into the two
//            byte words of the integer slicer;
//   phase 3  successor words by warp shuffle, cross product by one dp4a, sign bit shifted into a per-lane word
//            (bit = channel); two 32x32 bit-matrix transposes by shuffle turn them into per-channel
//            words (bit = time), which lanes OR into the global bit streams (natural sample order).
// ncu: profiles/.
#pragma once
#include "common.cuh"
#include "fft.cuh"

namespace snrx {

constexpr int kPfbD = 24;
constexpr int kTileT = 128;                    // channel-rate samples computed per tile
constexpr int kTileStride = 127;               // samples whose slicer bit the tile emits (needs y[m+1])
constexpr int kChunkT = 8;                     // output times per FIR lane and pass
constexpr int kVStride = 33;                   // float2 per row of a warp's V[48][32] tile (odd: conflict free)
constexpr float kMagic = 12582912.0f;          // 1.5 * 2^23: (x + kMagic) - kMagic == rint(x)

// BLE bank: even bin 2q (q = 0..47) -> BLE channel number, or -1 (bins +-41..+-47 MHz carry no channel)
SNRX_HD constexpr int ble_channel_of_q(int q) {
    int mhz = (q <= 23) ? 2440 + 2 * q : 2440 + 2 * (q - 48);
    if (mhz < 2402 || mhz > 2480) return -1;
    int k = (mhz - 2402) / 2;                  // RF channel index 0..39
    return k == 0 ? 37 : k <= 11 ? k - 1 : k == 12 ? 38 : k <= 38 ? k - 2 : 39;   // btle_rx.c:932-948 inverted
}

// position (in float2 units) of tile sample i' inside the skewed shared-memory tile: a 64-byte
// skew every 24*TT samples (TT = output times per FIR thread) keeps the FIR loads conflict free
template <int TT>
SNRX_HD constexpr int xs_pos(int ip) { return ip + 8 * ((ip + 12) / (24 * TT)); }

template <int NT, int TT = 16, int T = kTileT> struct PfbGeom {
    static constexpr int kHist = 24 * NT;                              // L: 384 or 768
    static constexpr int kTileIn = kHist + kPfbD * (T - 1) + 2;        // samples i' = 0 .. kTileIn-1 (even count)
    static constexpr int kPieces = (kTileIn + 12 + 24 * TT - 1) / (24 * TT);   // skew periods touched
    static constexpr int kXsLen = xs_pos<TT>(kTileIn) + 8;             // float2
};

// BLE kernel: one warp per CTA, 32 output times, 31 emitted decisions
template <int NT> struct PfbBleGeom {
    static constexpr int kT = 32;                                      // channel-rate samples computed per tile
    static constexpr int kStride = 31;                                 // samples whose slicer bit the tile emits
    static constexpr int kThreads = 32;
    using G = PfbGeom<NT, kChunkT, kT>;
    static constexpr int kXsBytes = ((G::kXsLen * 8 + 15) / 16) * 16;
    static constexpr int kVBytes = 8 * 32 * 16;                        // V[8][32] float4 = (branch r2 = rl, r2 = rl + 8) of one pass
    static constexpr int kSmemBytes = kXsBytes + kVBytes + 16;         // + the staging mbarrier
#ifndef SNRX_PFB_CTAS
#define SNRX_PFB_CTAS 16
#endif
    static constexpr int kCtasPerSm = (228 * 1024) / (kSmemBytes + 1024) < SNRX_PFB_CTAS ? (228 * 1024) / (kSmemBytes + 1024) : SNRX_PFB_CTAS;
};

// FIR of one thread.  xb = &xs[xs_pos-base of this thread], see fir_base().  acc[a][e] accumulates
// branch rho + 24 a at output time 16 q + e.
template <int NT, int A, int TT>
SNRX_HD void pfb_fir_thread(const float2* xb, int s0 /* 8 if rho <= 12 else 0 */, const float* g /*[NT]*/,
                            float2 (&acc)[A][TT]) {
    constexpr int kPer = 24 * TT;                     // skew period in samples
#pragma unroll
    for (int a = 0; a < A; a++)
#pragma unroll
        for (int e = 0; e < TT; e++) acc[a][e] = make_float2(0.f, 0.f);
#pragma unroll
    for (int u = -(NT - 1); u <= TT - 1; u++) {
        // skew of row u for rho >= 13 (floor((24u - 13 + 12)/kPer)), boundary rows add s0
        const int fl = (24 * u - 1 >= 0) ? (24 * u - 1) / kPer : -((-(24 * u - 1) + kPer - 1) / kPer);
        const int off = 24 * u + 8 * fl + ((u % TT == 0) ? s0 : 0);
        const float2 x = xb[off];
#pragma unroll
        for (int e = 0; e < TT; e++) {
            const int d = e - u;
            if (d >= 0 && d < NT) {
                acc[d % A][e] = f2_fma(make_float2(g[d], g[d]), x, acc[d % A][e]);
            }
        }
    }
}

// base pointer of FIR thread (rho, q): element u of pfb_fir_thread is tile sample
// i' = kHist + 24 TT q + 24 u - rho, stored at xs_pos<TT>(i')
template <int NT, int TT>
SNRX_HD int fir_base(int rho, int q) {
    return PfbGeom<NT, TT>::kHist + 24 * TT * q - rho + 8 * (PfbGeom<NT, TT>::kHist / (24 * TT) + q);
}

// Quantiser of the wideband path: q = clamp(rint(y * scale), -128, 127) evaluated as
//   u = sat(y * (scale/255) + 128/255)          one FFMA.SAT per component: the clamp is free
//   t = 1.5 * 2^23 + rint(255 u) - 128           255 u + (1.5 * 2^23 - 128), packed: t = 1.5 * 2^23 + q
// u carries one extra rounding (<= 2^-25, i.e. 8e-6 of a quantiser step): part of this engine's definition of
// its quantised channel streams (SNRX_STAGE_BLE_Q8), on which frame parity is stated (DESIGN.md 4).
// The kernel keeps the result biased: the slicer reads q from the bits of t (q8_of_biased, slicer_w / slicer_a).
SNRX_HD float2 quant_pair_biased(float2 y, float s255 /* +-scale/255, 0 beyond the capture end */) {
    const float ux = f_sat(f_fma(y.x, s255, 128.0f / 255.0f));
    const float uy = f_sat(f_fma(y.y, s255, 128.0f / 255.0f));
    return f2_fma(make_float2(ux, uy), make_float2(255.0f, 255.0f), make_float2(kMagic - 128.0f, kMagic - 128.0f));
}
// q itself as an integer-valued float (the Cooley-Tukey statement below)
SNRX_HD float2 quant_pair(float2 y, float s255) { return f2_add(quant_pair_biased(y, s255), make_float2(-kMagic, -kMagic)); }

SNRX_HD uint32_t f_bits(float x) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(x);
#else
    uint32_t u; memcpy(&u, &x, 4); return u;
#endif
}
// t = 1.5 * 2^23 + q, q in [-128, 127], lies in [2^23, 2^24) with unit spacing: its bits are 0x4B400000 + q, so byte 3 is
// always 0x4B and byte 0 is q as int8
SNRX_HD int8_t q8_of_biased(uint32_t t_bits) { return (int8_t)(t_bits & 0xFFu); }

// Bytes of the 64-bit value y:x picked by the selector nibbles of s (selector values 0..7 only)
SNRX_HD uint32_t byte_perm(uint32_t x, uint32_t y, uint32_t s) {
#ifdef __CUDA_ARCH__
    return __byte_perm(x, y, s);
#else
    const uint64_t v = ((uint64_t)y << 32) | x;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) r |= (uint32_t)((v >> (8 * ((s >> (4 * i)) & 7u))) & 0xFFu) << (8 * i);
    return r;
#endif
}
// Sum of the four products of the signed bytes of a and b
SNRX_HD int dp4a(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __dp4a((int)a, (int)b, 0);
#else
    int s = 0;
    for (int i = 0; i < 4; i++) s += (int)(int8_t)(a >> (8 * i)) * (int)(int8_t)(b >> (8 * i));
    return s;
#endif
}

// V tile of one FIR pass: row rl (0..7), column = output time, float4 = (branch r2 = rl, branch r2 = rl + 8)
// of the pass's 16-point transform; the column is XOR-swizzled with the row so that both the FIR lanes'
// stores (8 rows at one column) and the DFT lanes' loads (one row, 32 columns) are bank-conflict free.
SNRX_HD constexpr int v_pos(int row, int col) { return row * 32 + (col ^ row); }

// One lane's column of pass gi -> the 16 inputs of IdftPow2<16, 1>, in the prime-factor order of fft.cuh Pfa48: branch r2
// feeds input (r2 - Pfa48::rot(gi)) mod 16.  gi is a constant after unrolling, so the rotation is register naming only (as a
// template parameter ptxas allocated the phase worse: one 8-byte spill in k_pfb_ble<16, false>).
SNRX_HD void pfb_load_col16_pfa(const float4* V, int lane, int gi, cf (&v)[16]) {
    const int rot = Pfa48::rot(gi);
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const float4 t = V[v_pos(r, lane)];
        v[(r + 16 - rot) % 16].r = t.x; v[(r + 16 - rot) % 16].i = t.y;
        v[(r + 24 - rot) % 16].r = t.z; v[(r + 24 - rot) % 16].i = t.w;
    }
}

// Integer slicer on the quantiser's bits.  From t_i, t_q (bits of the biased I and Q of one sample), bytes low to high:
//   slicer_w = [I, ~Q, 0, 1]     (0x4B ^ 0x4B, 0x4B ^ 0x4A)    the word the PREDECESSOR sample reads
//   slicer_a = [Q, I, I, I]
// dp4a(slicer_a of sample m, slicer_w of sample m+1) = Q0 I1 + I0 (-Q1 - 1) + I0 * 0 + I0 = -(I0 Q1 - I1 Q0), exact: its sign
// bit is the decision b[m] = I0 Q1 - I1 Q0 > 0 (btle_rx.c:1357-1361).
SNRX_HD uint32_t slicer_w(uint32_t t_i, uint32_t t_q) { return byte_perm(t_i, t_q, 0x3340u) ^ 0x4A4BFF00u; }
SNRX_HD uint32_t slicer_a(uint32_t t_i, uint32_t t_q) { return byte_perm(t_i, t_q, 0x0004u); }
SNRX_HD uint32_t slicer_sign_dp4a(uint32_t a0, uint32_t w1) { return (uint32_t)dp4a(a0, w1); }
// the quantised (I, Q) back from slicer_a
SNRX_HD int8_t slicer_a_i(uint32_t a) { return (int8_t)(a >> 8); }
SNRX_HD int8_t slicer_a_q(uint32_t a) { return (int8_t)a; }

// Twiddle-free radix-3 combination of the three 16-point transforms (fft.cuh Pfa48) + rotation + quantisation:
// on return sw[q] / sa[q] hold slicer_w / slicer_a of the quantised (I, Q) of even bin 2q for the 40 bins that carry a BLE
// channel (the other 8 are never computed: dead code for the compiler).
// s_even / s_odd: quantiser scale with the sign of (-1)^(q m) folded in (0 beyond the capture end).
SNRX_HD void pfb_combine_quant_pfa(const cf (&f0)[16], const cf (&f1)[16], const cf (&f2)[16], uint32_t (&sw)[48],
                                   uint32_t (&sa)[48], float s_even, float s_odd, cf (&raw)[48], bool keep_raw) {
    cf y[48];
    Pfa48::template combine<0>(f0, f1, f2, y);
    const float se = f_mul(s_even, 1.0f / 255.0f), so = f_mul(s_odd, 1.0f / 255.0f);
#pragma unroll
    for (int q = 0; q < 48; q++) {
        if (ble_channel_of_q(q) < 0) { sw[q] = sa[q] = 0u; if (keep_raw) raw[q] = cf{0.f, 0.f}; continue; }
        if (keep_raw) raw[q] = y[q];
        const float2 t = quant_pair_biased(P(y[q]), (q & 1) ? so : se);
        sw[q] = slicer_w(f_bits(t.x), f_bits(t.y));
        sa[q] = slicer_a(f_bits(t.x), f_bits(t.y));
    }
}

// ---- The same phases 1-3 in their Cooley-Tukey form (twiddled radix-3 combination, float slicer): the statement the kernel
// ran before the prime-factor map.  The kernel no longer calls these; the CPU tile harness tests/emu/emu.cu steps them against
// the oracle, and tests/test_pfb_factored.py checks the kernel's path above against them tile by tile.
SNRX_HD void pfb_load_col16(const float4* V, int lane, cf (&v)[16]) {          // natural order r2 = n2
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const float4 t = V[v_pos(r, lane)];
        v[r].r = t.x; v[r].i = t.y; v[r + 8].r = t.z; v[r + 8].i = t.w;
    }
}
// on return y[q] holds the quantised (I, Q) of even bin 2q as integer-valued floats for the 40 bins that carry a BLE channel
SNRX_HD void pfb_combine_quant(const cf (&f0)[16], const cf (&f1)[16], const cf (&f2)[16], cf (&y)[48], float s_even,
                               float s_odd, cf (&raw)[48], bool keep_raw) {
    Idft3xQ<48>::template combine<0>(f0, f1, f2, y);
    const float se = f_mul(s_even, 1.0f / 255.0f), so = f_mul(s_odd, 1.0f / 255.0f);
#pragma unroll
    for (int q = 0; q < 48; q++) {
        if (ble_channel_of_q(q) < 0) { y[q] = cf{0.f, 0.f}; if (keep_raw) raw[q] = cf{0.f, 0.f}; continue; }
        if (keep_raw) raw[q] = y[q];
        y[q] = C(quant_pair(P(y[q]), (q & 1) ? so : se));
    }
}
// decision b[m] = I[m] Q[m+1] - I[m+1] Q[m] > 0 as the sign bit of 0.5 - cross: the operands are integers of magnitude <= 128,
// so 0.5 - cross is exact and never zero
SNRX_HD uint32_t slicer_sign(float i0, float q0, float i1, float q1) { return f_bits(f_fma(i1, q0, f_fma(-i0, q1, 0.5f))); }

// The 40 used bins in the order the slicer packs them: slot L of word A (L = 0..23) and of word B (L = 0..15)
SNRX_HD constexpr int ble_q_of_slot_a(int L) { return L < 21 ? L : L + 8; }     // q = 0..20, 29..31
SNRX_HD constexpr int ble_q_of_slot_b(int L) { return 32 + L; }                 // q = 32..47
// ble_channel_of_q(ble_q_of_slot_x(L)) as a handful of selects (the lanes of a tile need it at run time, where the general
// function costs four branches); checked against it below for every slot
SNRX_HD constexpr int ble_channel_of_slot_a(int L) { return L <= 19 ? 17 + L : L == 20 ? 39 : L == 21 ? 37 : L - 22; }
SNRX_HD constexpr int ble_channel_of_slot_b(int L) { return L <= 8 ? 2 + L : L == 9 ? 38 : 1 + L; }
constexpr bool ble_slot_channels_agree() {
    for (int L = 0; L < 24; L++) if (ble_channel_of_slot_a(L) != ble_channel_of_q(ble_q_of_slot_a(L))) return false;
    for (int L = 0; L < 16; L++) if (ble_channel_of_slot_b(L) != ble_channel_of_q(ble_q_of_slot_b(L))) return false;
    return true;
}
static_assert(ble_slot_channels_agree(), "slot -> BLE channel shortcut");

SNRX_HD uint32_t shift_in_sign(uint32_t acc, uint32_t sign_word) {   // (acc << 1) | (sign_word >> 31): one SHF
#ifdef __CUDA_ARCH__
    return __funnelshift_l(sign_word, acc, 1);
#else
    return (acc << 1) | (sign_word >> 31);
#endif
}

// One step of the 32x32 bit-matrix transpose across a warp (rows = lanes, columns = bits): exchange with
// lane ^ j the off-diagonal j x j blocks.  m = columns whose bit j is clear.
SNRX_HD uint32_t transpose_step(uint32_t x, uint32_t y /* value of lane ^ j */, int lane, int j, uint32_t m) {
#ifdef __CUDA_ARCH__
    // the same value with one rotate and one bitwise select: under m no bit of y >> j wraps, under ~m none of y << j does, so
    // both are rotations of y; keep = the bits this lane keeps.  (The two-sided form compiled to six predicated operations.)
    const bool hi = (lane & j) != 0;
    const uint32_t keep = hi ? ~m : m;
    const uint32_t r = __funnelshift_r(y, y, hi ? j : 32 - j);
    return (x & keep) | (r & ~keep);
#else
    return (lane & j) ? ((x & ~m) | ((y >> j) & m)) : ((x & m) | ((y << j) & ~m));
#endif
}

#if defined(__CUDACC__)

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::);
}

__device__ __forceinline__ void cp_async16_full(void* smem_dst, const void* gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc));
}

// ---- bulk (TMA) staging: one cp.async.bulk per skew piece, completion on an mbarrier.  The bytes go
// L2 -> shared memory through the async proxy: no LSU wavefronts, no per-lane address arithmetic.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool elect_one() {              // one lane of the (converged) warp
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Interior tile (entirely inside the capture): lane p < kPieces copies piece p -- tile samples
// i' in [24 TT p - 12, 24 TT (p+1) - 12) clipped to [0, kTileIn), stored at i' + 8 p.  All sizes and
// addresses are multiples of 16 bytes (kTileIn, 24 TT and the tile origin are even).
template <class G, int TT, bool INIT = false>
__device__ __forceinline__ void pfb_stage_tile_bulk(float2* xs, const float2* xtile /* sample i' = 0 */, uint64_t* bar, int lane) {
    constexpr int kPer = 24 * TT;
    static_assert(G::kPieces <= 32 && G::kTileIn % 2 == 0, "one lane per piece");
    // the barrier has count 1 and the tile is one phase of it.  ONE elected lane issues all the
    // copies (compile-time offsets and sizes, warp-uniform addresses): with one lane per piece the compiler serialises them
    // anyway -- a bulk copy takes its operands from uniform registers, so it elects a lane, broadcasts that lane's operands,
    // issues, and loops (ELECT / R2UR / UBLKCP / BRA.U.ANY six times in the sampled profile).
    (void)lane;
    if (elect_one()) {
        if (INIT) mbar_init(bar, 1);                      // a one-tile CTA: the elected lane also initialises the barrier (the
                                                          // caller's __syncwarp() before the wait publishes it to the other lanes)
        mbar_expect_tx(bar, (uint32_t)(G::kTileIn * sizeof(float2)));
#pragma unroll
        for (int p = 0; p < G::kPieces; p++) {
            const int lo = p == 0 ? 0 : kPer * p - 12;
            const int hi = kPer * (p + 1) - 12 < G::kTileIn ? kPer * (p + 1) - 12 : G::kTileIn;
            bulk_g2s(xs + lo + 8 * p, xtile + lo, (uint32_t)((hi - lo) * sizeof(float2)), bar);
        }
    }
}

// Stage tile samples i' = 0 .. kTileIn-1 (capture samples x0 + i') into the skewed tile: piece p holds
// i' in [24 TT p - 12, 24 TT (p+1) - 12) at position i' + 8 p; 16-byte copies (one sample pair each).
// Interior tiles (the whole tile inside the capture) take a fully unrolled path whose offsets are
// compile-time constants; tiles that touch either end of the capture zero-fill through the generic loop.
template <class G, int TT, int THREADS>
__device__ __forceinline__ void pfb_stage_tile(float2* xs, const float2* xcap, int64_t x0, int64_t n_in, int tid) {
    constexpr int kPer = 24 * TT, kPairs = kPer / 2;
    if (x0 >= 0 && x0 + G::kTileIn <= n_in) {
        if constexpr (THREADS % kPairs == 0) {
            constexpr int R = THREADS / kPairs;                 // pieces covered per sweep of the CTA
            const int pp = tid / kPairs, t = tid - pp * kPairs;
            const int ip_t = kPer * pp - 12 + 2 * t;            // this thread's i' in sweep 0
            const float2* src = xcap + x0 + ip_t;
            float2* dst = xs + ip_t + 8 * pp;
#pragma unroll
            for (int k = 0; k * R < G::kPieces; k++) {
                const int ip = ip_t + kPer * R * k;
                const bool ok = (k > 0 || ip >= 0) && ((k + 1) * R * kPer - 12 <= G::kTileIn || ip < G::kTileIn);
                if (ok) cp_async16_full(dst + (kPer + 8) * R * k, src + kPer * R * k);
            }
        } else {
            const float2* src = xcap + x0 + 2 * tid;
            float2* dst = xs + 2 * tid;
#pragma unroll
            for (int p = 0; p < G::kPieces; p++) {
#pragma unroll
                for (int t0 = 0; t0 < kPairs; t0 += THREADS) {
                    constexpr int dummy = 0; (void)dummy;
                    const int ip0 = kPer * p - 12 + 2 * t0;      // compile-time; this thread copies i' = ip0 + 2 tid
                    bool ok = true;
                    if (t0 + THREADS > kPairs) ok = ok && (t0 + tid < kPairs);
                    if (ip0 < 0) ok = ok && (ip0 + 2 * tid >= 0);
                    if (ip0 + 2 * (THREADS - 1) >= G::kTileIn) ok = ok && (ip0 + 2 * tid < G::kTileIn);
                    if (ok) cp_async16_full(dst + ip0 + 8 * p, src + ip0);
                }
            }
        }
        return;
    }
    for (int idx = tid; idx < G::kPieces * kPairs; idx += THREADS) {
        const int p = idx / kPairs, t = idx - p * kPairs;
        const int ip = kPer * p - 12 + 2 * t;
        if (ip >= 0 && ip < G::kTileIn) {
            const int64_t i = x0 + ip;
            const bool ok = (i >= 0) && (i + 1 < n_in);
            cp_async16(xs + ip + 8 * p, xcap + (ok ? i : 0), ok);
        }
    }
}

struct PfbBleArgs {
    const float2* x;          // [n_captures][stride] cf32
    uint64_t stride;          // samples between captures
    int64_t n_in;             // samples per capture
    int32_t n_out;            // channel-rate samples per capture (n_in / 24)
    int32_t n_tiles;          // tiles per capture in this launch
    int32_t tile0;            // first tile of this launch
    int32_t n_caps;           // captures in this launch
    const float4* taps_pass;  // [3][NT/4][8] float4: element (gi, d4, rl) = h[rho + 24 (4 d4 + 0..3)], rho = gi + 3 rl --
                              // the 8 FIR rows of a pass read 128 contiguous bytes per load
    float scale;              // quantiser scale
    uint32_t* bits;           // zero-initialised; tiles OR their words in
    BitsLayout lay;
    int8_t* dbg_q8;           // [cap][40][n_out][2] or null
    float2* dbg_cf;           // [cap][40][n_out] or null
};

// whether the tile is staged by bulk copies (it lies entirely inside the capture) or by the zero-filling generic path
template <class G>
SNRX_HD bool pfb_tile_interior(int64_t x0, int64_t n_in) { return x0 >= 0 && x0 + G::kTileIn <= n_in; }

// One tile, staged in xs, through phases 1-3.
template <int NT, bool DEBUG>
__device__ __forceinline__ void pfb_ble_tile(const PfbBleArgs& a, const float2* xs, float4* V, int lane, int cap, int g_first) {
    using B = PfbBleGeom<NT>;
    // ---- phase 1: three passes of FIR (branches r = gi mod 3) -> transpose -> 16-point inverse DFT
    cf f[3][16];
    {
        const int rl = lane & 7, c = lane >> 3;                            // c: chunk of 8 output times
#pragma unroll
        for (int gi = 0; gi < 3; gi++) {
            const int rho = gi + 3 * rl;
            float g[NT];
            const float4* gp = a.taps_pass + gi * (NT / 4) * 8 + rl;
#pragma unroll
            for (int d = 0; d < NT / 4; d++) {
                const float4 t = __ldg(gp + 8 * d);
                g[4 * d] = t.x; g[4 * d + 1] = t.y; g[4 * d + 2] = t.z; g[4 * d + 3] = t.w;
            }
            float2 acc[2][kChunkT];
            pfb_fir_thread<NT, 2, kChunkT>(xs + fir_base<NT, kChunkT>(rho, c), rho <= 12 ? 8 : 0, g, acc);
#pragma unroll
            for (int e = 0; e < kChunkT; e++)
                V[v_pos(rl, 8 * c + e)] = make_float4(acc[0][e].x, acc[0][e].y, acc[1][e].x, acc[1][e].y);
            __syncwarp();
            cf v16[16];
            pfb_load_col16_pfa(V, lane, gi, v16);
            __syncwarp();                                                  // V is rewritten by the next pass
            IdftPow2<16, 1>::run(v16, f[gi]);
        }
    }

    // ---- phase 2: radix-3 combination + rotation + quantiser + slicer words, one lane per output time
    uint32_t sw[48], sa[48];
    const int mg = g_first + lane;                           // channel-rate sample index in the capture
    {
        const float s = (mg < a.n_out) ? a.scale : 0.0f;
        cf raw[48];
        pfb_combine_quant_pfa(f[0], f[1], f[2], sw, sa, s, (mg & 1) ? -s : s, raw, DEBUG);
        if (DEBUG && lane < B::kStride && mg < a.n_out) {
#pragma unroll
            for (int qq = 0; qq < 48; qq++) {
                const int ch = ble_channel_of_q(qq);
                if (ch >= 0) {
                    const size_t o = ((size_t)cap * 40 + ch) * (size_t)a.n_out + mg;
                    if (a.dbg_q8) { a.dbg_q8[2 * o] = slicer_a_i(sa[qq]); a.dbg_q8[2 * o + 1] = slicer_a_q(sa[qq]); }
                    if (a.dbg_cf) {
                        const float sg = ((qq & 1) && (mg & 1)) ? -1.0f : 1.0f;
                        a.dbg_cf[o] = make_float2(raw[qq].r * sg, raw[qq].i * sg);
                    }
                }
            }
        }
    }

    // ---- phase 3: slicer bits (btle_rx.c:1357-1361), transposed to one word per channel, OR-ed into the streams
    {
        uint32_t wa = 0, wb = 0;                             // bit L = decision of slot L (ble_q_of_slot_a / _b) at time `lane`
#pragma unroll
        for (int L = 23; L >= 0; L--) {
            const int qq = ble_q_of_slot_a(L);
            wa = shift_in_sign(wa, slicer_sign_dp4a(sa[qq], __shfl_down_sync(0xffffffffu, sw[qq], 1)));
        }
#pragma unroll
        for (int L = 15; L >= 0; L--) {
            const int qq = ble_q_of_slot_b(L);
            wb = shift_in_sign(wb, slicer_sign_dp4a(sa[qq], __shfl_down_sync(0xffffffffu, sw[qq], 1)));
        }
        // rows = times (lanes), columns = slots  ->  rows = slots, columns = times
        {
            const uint32_t o = __shfl_xor_sync(0xffffffffu, wb, 16);
            wb = (wb & 0xFFFFu) | (o << 16);                 // lanes 0..15: times 0..15 | times 16..31 of slots 0..15
        }
        wa = transpose_step(wa, __shfl_xor_sync(0xffffffffu, wa, 16), lane, 16, 0x0000FFFFu);
        // written out: as a `for (j = 8; j >= 1; j >>= 1)` loop ptxas kept it rolled (shift counts and masks in registers, a
        // branch per step: the sampled profile had the four steps at 4 % of the warp time)
#define SNRX_TRANSPOSE_STEP(J, M)                                                       \
        wa = transpose_step(wa, __shfl_xor_sync(0xffffffffu, wa, J), lane, J, M);       \
        wb = transpose_step(wb, __shfl_xor_sync(0xffffffffu, wb, J), lane, J, M);
        SNRX_TRANSPOSE_STEP(8, 0x00FF00FFu)
        SNRX_TRANSPOSE_STEP(4, 0x0F0F0F0Fu)
        SNRX_TRANSPOSE_STEP(2, 0x33333333u)
        SNRX_TRANSPOSE_STEP(1, 0x55555555u)
#undef SNRX_TRANSPOSE_STEP
        // lane L now holds the 32 decisions (bit = time) of slot L; the tile's last sample has no successor in it
        const uint32_t wi = (uint32_t)kBitsLeadWords + ((uint32_t)g_first >> 5);
        const int off = g_first & 31;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            const uint32_t mk = (half ? wb : wa) & 0x7FFFFFFFu;
            if (lane < (half ? 16 : 24) && mk) {
                const int ch = half ? ble_channel_of_slot_b(lane) : ble_channel_of_slot_a(lane);
                uint32_t* dst = a.bits + a.lay.index(cap, ch, wi);
                atomicOr(dst, mk << off);
                if (off > 1 && (mk >> (32 - off))) atomicOr(dst + 1, mk >> (32 - off));
            }
        }
    }
}

// One tile per one-warp CTA: any tile (interior tiles by bulk copies, tiles that touch either end of the capture through the
// zero-filling generic path).
// Grid = (tiles of the launch, captures): the tile's input address needs no division, so the bulk copies leave a few dozen
// instructions after the CTA starts (the sampled profile of the 1-D grid had 7 % of the warp time in the index arithmetic
// ahead of the copy: two 32-bit divisions through the conversion unit).  Measured and rejected: two / four warps per CTA
// (independent tiles, fewer CTAs for the block scheduler to start): 0.337 / 0.341 ms against 0.330.
template <int NT, bool DEBUG>
__global__ void __launch_bounds__(32, PfbBleGeom<NT>::kCtasPerSm) k_pfb_ble(PfbBleArgs a) {
    using B = PfbBleGeom<NT>;
    using G = typename B::G;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* xs = reinterpret_cast<float2*>(smem_raw);
    float4* V = reinterpret_cast<float4*>(smem_raw + B::kXsBytes);         // [8][32], see v_pos()
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + B::kXsBytes + B::kVBytes);

    int lane = threadIdx.x;
    asm volatile("" : "+r"(lane));                         // opaque: ptxas re-read SR_TID.X (S2R + a dependent shift chain) in mid-tile
    const int tile = a.tile0 + (int)blockIdx.x;
    const int cap = (int)blockIdx.y;
    const float2* xcap = a.x + (size_t)cap * a.stride;
    const int g_first = B::kStride * tile;                                 // first channel sample of the tile

    // ---- phase 0: stage the input tile (bulk copies for interior tiles, zero-filling cp.async at the capture ends)
    const int64_t x0 = (int64_t)kPfbD * g_first - G::kHist;
    // (an L2 prefetch of the input a CTA `n` launches behind this one will stage -- cp.async.bulk.prefetch.L2, 1184 ... 9472 tiles
    // ahead -- was measured: 0.333 / 0.334 / 0.336 / 0.336 / 0.338 ms, no gain: what a fresh CTA waits for is not HBM-vs-L2 latency)
    if (pfb_tile_interior<G>(x0, a.n_in)) {
        pfb_stage_tile_bulk<G, kChunkT, true>(xs, xcap + x0, bar, lane);
        __syncwarp();
        mbar_wait(bar, 0);
    } else {
        pfb_stage_tile<G, kChunkT, B::kThreads>(xs, xcap, x0, a.n_in, lane);
        cp_async_commit_wait_all();
        __syncwarp();
    }
    pfb_ble_tile<NT, DEBUG>(a, xs, V, lane, cap, g_first);
}

#endif  // __CUDACC__

}  // namespace snrx
