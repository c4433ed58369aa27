// frame_rf.cuh -- radio metrics of every decoded frame (include/snoutrx.h snrx_frame_rf_t): signal power, noise floor, SNR
// and carrier offset, recomputed from the batch's input over two short windows per frame.
//
// The channel samples of a frame exist nowhere else: the wideband channelizers turn the input straight into slicer bits /
// discriminator output.  k_frame_rf evaluates the channelizer definition for the frame's one bin, which factors into
// "mix, then a real FIR":
//   y_k[m] = (-j)^(k m) sum_n h[n] W^(k n) x[24 m - n] = sum_n h[n] (exp(-j 2 pi k i / 96) x[i]),  i = 24 m - n
// so every staged input sample is mixed once and every tap costs 2 FMAs.  The buffer index i equals the capture index
// modulo 96 (shard pre halos are multiples of 128 channel samples = 3072 input samples), so the mix is the capture's.
// Narrow-band frames read y = x directly.
//
// The arithmetic of a window (power and lag-1 sums, the FIR of one output, theta0 of the 40 known BLE bits) is in
// __host__ __device__ cores that tests/emu steps on the CPU.
#pragma once
#include "common.cuh"
#include "synth.cuh"

namespace snrx {

static_assert(sizeof(snrx_frame_rf_t) == 40, "snrx_frame_rf_t layout (include/snoutrx.h, _abi.RF_DTYPE)");
constexpr int kRfWarps = 8;                // frames in flight per CTA (one warp each)
constexpr int kRfChunk = 32;                // channel samples per FIR pass: one per lane
constexpr double kRfFs = 4.0e6;
constexpr int kRfBleRefOrigin = -39;        // first sample of the reference GFSK burst, relative to sample_index
constexpr int kRfBleRefFirst = -24 - kRfBleRefOrigin, kRfBleRefEnd = 120 - kRfBleRefOrigin;   // burst samples of the window

// signal and noise windows of a frame, capture-relative channel indices (include/snoutrx.h)
struct RfWin { int64_t a, b; };
SNRX_HD void rf_windows(int proto, int64_t s, RfWin& sig, RfWin& noise) {
    if (proto == SNRX_PROTO_BLE) { sig.a = s - 24; sig.b = s + 120; noise.a = s - 104; noise.b = s - 40; }
    else { sig.a = s - 392; sig.b = s - 136; noise.a = s - 720; noise.b = s - 656; }
}
SNRX_HD int rf_bin(int proto, int channel) {
    return pfb_bin_of_mhz(proto == SNRX_PROTO_BLE ? ble_channel_mhz(channel) : zb_channel_mhz(channel));
}

// the 40 known bits of a BLE frame, LSB = first: preamble (0xAA, or 0x55 when AA bit 0 is 1), then the access address
SNRX_HD uint64_t rf_ble_known_bits(uint32_t aa) { return (uint64_t)((aa & 1u) ? 0x55u : 0xAAu) | ((uint64_t)aa << 8); }
// phase increment (rad) of the zero-offset reference burst from sample i - 1 to sample i (1 <= i)
SNRX_HD double rf_ble_dtheta(uint64_t bits, const double* gauss, int i) {
    return kGfskPhasePerFreq * gfsk_freq(gauss, (int64_t)i - 1, 40, [&](int64_t j) { return (int)((bits >> j) & 1u); });
}

// running sums of a window: sum |y|^2 and sum y[m] conj(y[m-1])
struct RfAcc { float p, lr, li; };
SNRX_HD void rf_acc_power(RfAcc& a, float2 y) { a.p = f_fma(y.x, y.x, f_fma(y.y, y.y, a.p)); }
SNRX_HD void rf_acc_lag(RfAcc& a, float2 y, float2 yp) {
    a.lr = f_fma(y.x, yp.x, f_fma(y.y, yp.y, a.lr));
    a.li = f_fma(y.y, yp.x, f_fma(-y.x, yp.y, a.li));
}
SNRX_HD float rf_db(float sum, int n) {
    const float mean = sum / (float)n;
    return mean < 1e-20f ? -200.0f : 10.0f * log10f(mean);
}
// fs / 2 pi * wrap(arg(lag) - theta0), wrap to [-pi, pi)
SNRX_HD float rf_cfo_hz(float lr, float li, double theta0) {
    const double two_pi = 6.283185307179586476925286766559;
    double d = atan2((double)li, (double)lr) - theta0;
    d -= two_pi * floor((d + 0.5 * two_pi) / two_pi);
    return (float)(d * (kRfFs / two_pi));
}

// One wideband output: y = sum_{d < NT} sum_{r < 24} h[24 d + r] P[r][c0 - d], where P[r][c] = mixed x[24 (q0 + c) - r] and
// c0 = the output's column.  P rows are `pst` float2 apart.
SNRX_HD float2 rf_fir(const float2* P, int pst, const float* h, int nt, int c0) {
    float ar = 0.0f, ai = 0.0f;
    for (int d = 0; d < nt; d++) {
        const float2* col = P + (c0 - d);
        const float* hd = h + 24 * d;
#pragma unroll
        for (int r = 0; r < 24; r++) {
            const float2 v = col[r * pst];
            ar = f_fma(hd[r], v.x, ar);
            ai = f_fma(hd[r], v.y, ai);
        }
    }
    return make_float2(ar, ai);
}
// mixed input sample: exp(-j 2 pi k i / 96) x[i], from the table w96[t] = exp(-j 2 pi t / 96); i96 = i mod 96
SNRX_HD float2 rf_mix(float2 x, const float2* w96, int k, int i96) {
    const float2 w = w96[(k * i96) % 96];
    return make_float2(f_fma(x.x, w.x, -(x.y * w.y)), f_fma(x.x, w.y, x.y * w.x));
}

// columns of P: 31 + nt (odd for nt = 16, 32, so a warp's stores along r hit distinct banks)
SNRX_HD int rf_cols(int nt) { return kRfChunk - 1 + nt; }

#if defined(__CUDACC__)
struct RfArgs {
    const float2* x; uint64_t stride;   // cf32 input the front end read, captures `stride` samples apart
    int64_t n_in;                       // input samples per capture in the buffer
    int32_t n_out;                      // channel samples per capture in the buffer
    int32_t nt;                         // wideband: taps per polyphase branch (16 / 32); 0 = narrow band
    int64_t origin;                     // capture-relative channel index of buffer sample 0 (first_window * 8192 - pre halo)
    uint32_t first_capture;
    const float* taps_ble; const float* taps_zb;   // wideband prototypes (24 * nt floats; null if the protocol is absent)
    const double* gauss;                // [16] Gaussian taps of the GFSK reference
    const snrx_frame_t* frames; const uint32_t* totals; uint32_t frame_cap;
    snrx_frame_rf_t* out;
};

// Sums of one window [a, b) (buffer-local) of one frame, by one warp.  lag: also the lag-1 products over [a, b), which read
// y[a - 1].  Every lane returns the warp's total.
__device__ inline RfAcc rf_window_warp(const RfArgs& A, const float2* xc, const float2* w96, const float* h, int k, float2* P,
                                       int64_t a, int64_t b, bool lag) {
    const int lane = threadIdx.x & 31;
    RfAcc acc{0.0f, 0.0f, 0.0f};
    float2 carry = make_float2(0.0f, 0.0f);
    const int pst = rf_cols(A.nt);
    for (int64_t m0 = a - (lag ? 1 : 0); m0 < b; m0 += kRfChunk) {
        const int64_t m = m0 + lane;
        float2 y = make_float2(0.0f, 0.0f);
        if (A.nt == 0) {
            if (m < b) y = xc[m];
        } else {
            // stage the mixed input of outputs m0 .. m0 + 31: P[r][c] = x~[24 (q0 + c) - r], q0 = m0 - nt + 1
            const int64_t i0 = 24 * (m0 - A.nt + 1) - 23;
            const int r0 = (int)((i0 % 96 + 96) % 96), n = 24 * pst;    // 32-bit residues inside the tile
            __syncwarp();
            for (int e = lane; e < n; e += 32) {
                const int64_t i = i0 + e;
                float2 v = make_float2(0.0f, 0.0f);
                if (i >= 0 && i < A.n_in) v = rf_mix(xc[i], w96, k, (r0 + e) % 96);
                P[(23 - e % 24) * pst + e / 24] = v;
            }
            __syncwarp();
            y = rf_fir(P, pst, h, A.nt, lane + A.nt - 1);
        }
        float2 yp = make_float2(__shfl_up_sync(0xffffffffu, y.x, 1), __shfl_up_sync(0xffffffffu, y.y, 1));
        if (lane == 0) yp = carry;
        carry = make_float2(__shfl_sync(0xffffffffu, y.x, 31), __shfl_sync(0xffffffffu, y.y, 31));
        if (m >= a && m < b) {
            rf_acc_power(acc, y);
            if (lag) rf_acc_lag(acc, y, yp);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        acc.p += __shfl_xor_sync(0xffffffffu, acc.p, o);
        acc.lr += __shfl_xor_sync(0xffffffffu, acc.lr, o);
        acc.li += __shfl_xor_sync(0xffffffffu, acc.li, o);
    }
    return acc;
}

// One warp per frame, grid-stride over the device-side frame count (no host round trip).  Shared memory: the mix table,
// one P tile per warp and the two prototypes (wideband only).
__global__ void __launch_bounds__(32 * kRfWarps) k_frame_rf(const RfArgs A) {
    extern __shared__ __align__(16) float2 rf_smem[];
    float2* w96 = rf_smem;
    for (int t = threadIdx.x; t < 96; t += blockDim.x) {
        float s, c;
        sincospif((float)t / 48.0f, &s, &c);
        w96[t] = make_float2(c, -s);
    }
    const int L = 24 * A.nt;
    float* taps = reinterpret_cast<float*>(rf_smem + 96 + (size_t)kRfWarps * 24 * rf_cols(A.nt));   // [BLE | 802.15.4]
    for (int t = threadIdx.x; t < L; t += blockDim.x) {
        taps[t] = A.taps_ble ? A.taps_ble[t] : 0.0f;
        taps[L + t] = A.taps_zb ? A.taps_zb[t] : 0.0f;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float2* P = rf_smem + 96 + (size_t)warp * 24 * rf_cols(A.nt);
    uint32_t n = A.totals[0] + A.totals[2];
    if (n > A.frame_cap) n = A.frame_cap;
    const float qnan = __int_as_float(0x7fc00000);
    for (uint32_t fi = blockIdx.x * kRfWarps + warp; fi < n; fi += gridDim.x * kRfWarps) {
        const snrx_frame_t& f = A.frames[fi];
        const int proto = f.proto;
        const int64_t s = f.sample_index;
        RfWin sig, noise;
        rf_windows(proto, s, sig, noise);
        const int64_t cap = (int64_t)f.capture_id - A.first_capture;
        const float2* xc = A.x + (size_t)cap * A.stride;
        const float* h = proto == SNRX_PROTO_BLE ? taps : taps + L;
        const int k = rf_bin(proto, f.channel);
        // windows in the capture and in the buffer; the signal window also reads y[a - 1]
        const bool sig_ok = sig.a - 1 >= 0 && sig.a - 1 - A.origin >= 0 && sig.b - A.origin <= A.n_out;
        const bool noise_ok = noise.a >= 0 && noise.a - A.origin >= 0 && noise.b - A.origin <= A.n_out;
        RfAcc as{0.0f, 0.0f, 0.0f}, an{0.0f, 0.0f, 0.0f};
        if (sig_ok) as = rf_window_warp(A, xc, w96, h, k, P, sig.a - A.origin, sig.b - A.origin, true);
        if (noise_ok) an = rf_window_warp(A, xc, w96, h, k, P, noise.a - A.origin, noise.b - A.origin, false);
        double theta0 = SNRX_RF_ZB_THETA0;
        if (proto == SNRX_PROTO_BLE && sig_ok) {
            const uint64_t bits = rf_ble_known_bits(f.access_addr);
            double cr = 0.0, ci = 0.0;
            for (int i = kRfBleRefFirst + lane; i < kRfBleRefEnd; i += 32) {
                double sn, cs;
                sincos(rf_ble_dtheta(bits, A.gauss, i), &sn, &cs);
                cr += cs; ci += sn;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                cr += __shfl_xor_sync(0xffffffffu, cr, o);
                ci += __shfl_xor_sync(0xffffffffu, ci, o);
            }
            theta0 = atan2(ci, cr);
        }
        if (lane == 0) {
            snrx_frame_rf_t r;
            r.sample_index = s; r.capture_id = f.capture_id; r.frame = fi; r.channel = f.channel; r.proto = f.proto;
            r.valid = (uint8_t)((sig_ok ? SNRX_RF_POWER | SNRX_RF_CFO : 0) | (noise_ok ? SNRX_RF_NOISE : 0));
            r.power_dbfs = sig_ok ? rf_db(as.p, (int)(sig.b - sig.a)) : qnan;
            r.noise_dbfs = noise_ok ? rf_db(an.p, (int)(noise.b - noise.a)) : qnan;
            r.snr_db = sig_ok && noise_ok ? r.power_dbfs - r.noise_dbfs : qnan;
            r.cfo_hz = sig_ok ? rf_cfo_hz(as.lr, as.li, theta0) : qnan;
            r.reserved = 0;
            A.out[fi] = r;
        }
    }
}

inline size_t rf_smem_bytes(int nt) {
    return sizeof(float2) * (96 + (nt ? (size_t)kRfWarps * 24 * rf_cols(nt) : 0)) + sizeof(float) * 2 * 24 * (size_t)nt;
}
#endif

// the 16 Gaussian taps of the GFSK reference: rectangular symbol convolved with a Gaussian of BT = 0.5, 4 samples per
// symbol over 4 symbols (snout_b200/synth.py gaussian_taps)
inline void rf_gauss_taps(double* g) {
    const double a = 3.14159265358979323846 * 0.5 * std::sqrt(2.0 / std::log(2.0));
    for (int n = 0; n < 16; n++) {
        const double t = (n - 8) / 4.0;
        g[n] = 0.5 * (std::erf(a * (t + 0.5)) - std::erf(a * (t - 0.5)));
    }
}

}  // namespace snrx
