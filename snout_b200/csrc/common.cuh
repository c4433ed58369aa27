// common.cuh -- shared definitions of the libsnoutrx kernels.
//
// Every arithmetic core is written as a __host__ __device__ function so that
// tests/emu (an nvcc-built HOST harness, test infrastructure only) can step the
// same per-thread code on the CPU and compare it with the oracle before any GPU
// time is spent.  libsnoutrx.so itself contains no host execution path for
// them: the ABI launches kernels or fails.
#pragma once
#include <cstdint>
#include <cmath>
#include "../../include/snoutrx.h"

#if defined(__CUDACC__)
#define SNRX_HD __host__ __device__ __forceinline__
#define SNRX_D __device__ __forceinline__
#else
#define SNRX_HD inline
#define SNRX_D inline
#endif

namespace snrx {

// ---- explicitly rounded float ops: never contracted / re-associated, identical on host and device
SNRX_HD float f_fma(float a, float b, float c) {
#ifdef __CUDA_ARCH__
    return __fmaf_rn(a, b, c);
#else
    return fmaf(a, b, c);
#endif
}
SNRX_HD float f_mul(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    volatile float r = a * b; return r;
#endif
}
SNRX_HD float f_add(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    volatile float r = a + b; return r;
#endif
}
SNRX_HD float f_sub(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fsub_rn(a, b);
#else
    volatile float r = a - b; return r;
#endif
}
SNRX_HD float f_sat(float a) {             // clamp to [0, 1]; folds into the producing FFMA as .SAT on the device
#ifdef __CUDA_ARCH__
    return __saturatef(a);
#else
    return fminf(fmaxf(a, 0.0f), 1.0f);
#endif
}
SNRX_HD float f_div(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fdiv_rn(a, b);
#else
    volatile float r = a / b; return r;
#endif
}
// ---- packed pairs: sm_100 issues two FP32 operations on a 64-bit register pair as ONE instruction
// (PTX fma/add/mul.rn.f32x2 -> SASS FFMA2/FADD2/FMUL2; ptxas folds operand swaps, per-half negation and
// scalar broadcast into the instruction).  Same FP32-pipe time as two scalar ops but half the issue
// slots -- and the channelizer is issue bound.  Each half is an IEEE-754 round-to-nearest operation,
// so the host statement below (tests/emu) is bit-identical.
#if defined(__CUDACC__)
SNRX_HD float2 f2_fma(float2 a, float2 b, float2 c) {
#ifdef __CUDA_ARCH__
    unsigned long long ra, rb, rc, rd;
    float2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
#else
    return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#endif
}
SNRX_HD float2 f2_add(float2 a, float2 b) {
#ifdef __CUDA_ARCH__
    unsigned long long ra, rb, rd;
    float2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
#else
    return make_float2(f_add(a.x, b.x), f_add(a.y, b.y));
#endif
}
SNRX_HD float2 f2_mul(float2 a, float2 b) {
#ifdef __CUDA_ARCH__
    unsigned long long ra, rb, rd;
    float2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
#else
    return make_float2(f_mul(a.x, b.x), f_mul(a.y, b.y));
#endif
}
#endif

SNRX_HD double d_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}
SNRX_HD double d_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}

// ---- channel plan: centre frequencies (get_freq_by_channel_number, btle_rx.c:932-948; top_block.py:56) and the
// channelizer bin of a centre frequency (bin k sits at 2440 + k MHz, modulo 96 MHz)
SNRX_HD int ble_channel_mhz(int ch) {
    if (ch == 37) return 2402;
    if (ch == 38) return 2426;
    if (ch == 39) return 2480;
    if (ch >= 0 && ch <= 10) return 2404 + 2 * ch;
    if (ch >= 11 && ch <= 36) return 2428 + 2 * (ch - 11);
    return -1;
}
SNRX_HD int zb_channel_mhz(int ch) { return (ch >= 11 && ch <= 26) ? 2400 + 5 * (ch - 10) : -1; }
SNRX_HD int pfb_bin_of_mhz(int mhz) { return mhz < 0 ? -1 : ((mhz - 2440) % 96 + 96) % 96; }

// ---- BLE constants (vendor/BTLE/host/btle-tools/src/btle_rx.c) -------------------------------
constexpr int kSps = 4;                    // SAMPLE_PER_SYMBOL, btle_rx.c:176
constexpr int kWindow = SNRX_BLE_WINDOW;   // 8192 IQ per receiver() call, btle_rx.c:180-182, 2382
constexpr int kSpanInt8 = 31 * 8 + 16384;  // receiver() buf_len, btle_rx.c:2382
constexpr int kDemodLimitInt8 = 19392;     // demod_buf_len, btle_rx.c:2025
constexpr int kBleMaxBytes = 42;           // 2 header + 37 payload + 3 crc, btle_rx.c:1344
constexpr int kBitsLeadWords = 4;          // samples -128..-1: zeros (history of a search origin, btle_rx.c:1377)
constexpr int kBitsTailWords = 64;         // zero words after the capture: a frame at the very end reads
                                           // 4*(32+16+8*40) = 1472 samples = 46 words past its start

// Bit layout: one word stream per (capture, channel), samples in natural order: bit (n & 31) of word
// kBitsLeadWords + (n >> 5) is the slicer decision of channel-rate sample n.  Symbol-spaced decisions
// (stride 4 samples, btle_rx.c:1357-1361) are picked out where they are needed: by the funnel shifts of the
// sliding correlation and, per candidate, by symbols32().
struct BitsLayout {
    uint32_t words_per_stream;  // kBitsLeadWords + ceil(n_out / 32) + kBitsTailWords
    uint32_t n_channels;
    SNRX_HD size_t index(uint32_t cap, uint32_t ch, uint32_t w) const {
        return ((size_t)cap * n_channels + ch) * (size_t)words_per_stream + w;
    }
};
SNRX_HD constexpr uint32_t bits_words_for(uint32_t n_out) { return kBitsLeadWords + (n_out + 31) / 32 + kBitsTailWords; }

SNRX_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int sh) {      // bits sh .. sh+31 of hi:lo, 0 <= sh < 32
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}
// every 4th bit of x starting at bit 0 -> low 8 bits
SNRX_HD uint32_t compress4(uint32_t x) {
    x &= 0x11111111u;
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    x = (x | (x >> 12)) & 0x000000FFu;
    return x;
}
// 32 symbol decisions (every 4th sample) starting at channel-rate sample s >= -128, LSB = first symbol
SNRX_HD uint32_t symbols32(const uint32_t* stream_words, int s) {
    const int n = s + 32 * kBitsLeadWords, w = n >> 5, sh = n & 31;
    uint32_t r = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) r |= compress4(funnel_r(stream_words[w + q], stream_words[w + q + 1], sh)) << (8 * q);
    return r;
}

// An access-address hit found by the sliding correlation.
struct Cand {
    int32_t s;          // channel-rate sample index of AA bit 0 (local to the processed buffer)
    uint16_t ch_idx;    // channel slot (index into the engine's channel list)
    uint8_t vneed;      // low AA positions that do NOT match: 0 = full 32-bit match, v>0 = usable only at a
                        // search origin whose zeroed history covers the first v positions (btle_rx.c:1377)
    uint8_t pad;
    uint32_t cap;       // capture index inside the batch
};

// Speculative decode of a candidate (one warp per candidate).
struct Dec {
    int32_t s;
    int32_t resume;     // sample where the reference resumes searching after this hit
    uint8_t len;        // payload length field
    uint8_t emit;       // 1: a frame is printed (length gate passed / data channel)
    uint8_t crc_ok;
    uint8_t vneed;
    uint8_t bytes[44];  // de-whitened header | payload | crc
};

struct BleParams {
    uint32_t aa;
    uint32_t aa_mask;
    uint32_t crc_init_internal;   // crc_init_reorder(-k), btle_rx.c:1801-1825
    int32_t n_out;                // channel-rate samples per capture in this buffer
    int32_t m_origin;             // local sample index where window `first_window` starts (multiple of 128)
    int32_t n_windows;            // windows whose frames belong to this call
    uint32_t first_window;
    uint32_t first_capture;
    uint32_t n_captures;
    uint32_t n_channels;
};

}  // namespace snrx
