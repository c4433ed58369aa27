// TEST INFRASTRUCTURE ONLY.  Host-side stepping of k_frame_rf's __host__ __device__ cores (snout_b200/csrc/frame_rf.cuh),
// built by nvcc into a temporary shared library by tests/test_rf.py and run on the CPU (no GPU needed), so that the
// radio-metrics arithmetic is checked against oracle/rf_oracle.py before GPU time is spent.  Never part of libsnoutrx.so.
#include <cmath>
#include <vector>
#include "../../snout_b200/csrc/frame_rf.cuh"

using namespace snrx;

// ---- radio metrics (k_frame_rf's cores) -----------------------------------------------------------
extern "C" {

void emu_rf_gauss(double* g) { rf_gauss_taps(g); }
int emu_rf_bin(int proto, int channel) { return rf_bin(proto, channel); }
// signal and noise windows of a frame at sample_index s: out = {sig.a, sig.b, noise.a, noise.b}
void emu_rf_windows(int proto, int64_t s, int64_t* out) {
    RfWin sig, noise;
    rf_windows(proto, s, sig, noise);
    out[0] = sig.a; out[1] = sig.b; out[2] = noise.a; out[3] = noise.b;
}
double emu_rf_ble_theta0(uint32_t aa, const double* gauss) {
    const uint64_t bits = rf_ble_known_bits(aa);
    double cr = 0.0, ci = 0.0;
    for (int i = kRfBleRefFirst; i < kRfBleRefEnd; i++) { const double d = rf_ble_dtheta(bits, gauss, i); cr += cos(d); ci += sin(d); }
    return atan2(ci, cr);
}
// sums of a window over its channel samples y (cf32): with lag, y[0] is the sample before the window and y[1 .. n] the window
void emu_rf_sums(const float* y, int n, int lag, float* out) {
    RfAcc a{0.0f, 0.0f, 0.0f};
    const int o = lag ? 1 : 0;
    for (int m = 0; m < n; m++) {
        const float2 v = make_float2(y[2 * (m + o)], y[2 * (m + o) + 1]);
        rf_acc_power(a, v);
        if (lag) rf_acc_lag(a, v, make_float2(y[2 * (m + o - 1)], y[2 * (m + o - 1) + 1]));
    }
    out[0] = a.p; out[1] = a.lr; out[2] = a.li;
}
float emu_rf_db(float sum, int n) { return rf_db(sum, n); }
float emu_rf_cfo_hz(float lr, float li, double theta0) { return rf_cfo_hz(lr, li, theta0); }
// channel samples m in [m0, m1) of bin k (wideband): the kernel's staging of 32-sample chunks into P tiles, then rf_fir
void emu_rf_channel(const float* x, int64_t n_in, const float* h, int nt, int k, int64_t m0, int64_t m1, float* out) {
    float2 w96[96];
    for (int t = 0; t < 96; t++) w96[t] = make_float2((float)cos(2.0 * M_PI * t / 96), (float)-sin(2.0 * M_PI * t / 96));
    const int pst = rf_cols(nt);
    std::vector<float2> P((size_t)24 * pst);
    for (int64_t c0 = m0; c0 < m1; c0 += kRfChunk) {
        const int64_t i0 = 24 * (c0 - nt + 1) - 23;
        for (int e = 0; e < 24 * pst; e++) {
            const int64_t i = i0 + e;
            float2 v = make_float2(0.0f, 0.0f);
            if (i >= 0 && i < n_in) v = rf_mix(make_float2(x[2 * i], x[2 * i + 1]), w96, k, (int)(i % 96));
            P[(size_t)(23 - e % 24) * pst + e / 24] = v;
        }
        for (int lane = 0; lane < kRfChunk && c0 + lane < m1; lane++) {
            const float2 y = rf_fir(P.data(), pst, h, nt, lane + nt - 1);
            out[2 * (c0 + lane - m0)] = y.x; out[2 * (c0 + lane - m0) + 1] = y.y;
        }
    }
}

}  // extern "C"
