// fft.cuh -- fully unrolled in-register inverse DFTs (kernel exp(+j 2 pi k r / N)) for the
// channelizer: N = 3 * 2^p (48 for the even-bin BLE bank, 96 for the full bank).  Pfa48 is the twiddle-free
// prime-factor form of the 48-point transform that the BLE channelizer runs.
//
// Everything is resolved at compile time: the recursion is template recursion, all array
// indices are constants after unrolling (so the arrays live in registers) and the twiddles are
// constexpr values that end up as FFMA immediates.  Radix-2 decimation in time below a single
// radix-3 stage; butterflies use the form  out0 = E + w O, out1 = 2E - out0, written on (re, im) register
// pairs so that each complex multiply-add is 2-3 packed FFMA2 instructions (common.cuh f2_*).
#pragma once
#include "common.cuh"

namespace snrx {

struct cf { float r, i; };

namespace detail {
constexpr double kPi = 3.14159265358979323846264338327950288;

constexpr double cx_sin_small(double x) {   // |x| <= pi/4, Taylor to x^19
    double x2 = x * x, term = x, sum = x;
    for (int k = 1; k <= 9; ++k) { term *= -x2 / ((2 * k) * (2 * k + 1)); sum += term; }
    return sum;
}
constexpr double cx_cos_small(double x) {
    double x2 = x * x, term = 1.0, sum = 1.0;
    for (int k = 1; k <= 10; ++k) { term *= -x2 / ((2 * k - 1) * (2 * k)); sum += term; }
    return sum;
}
// cos / sin of 2*pi*num/den with exact octant reduction
constexpr double cx_cos_frac(int num, int den) {
    num %= den; if (num < 0) num += den;
    // reduce to the first octant using symmetries, working on the fraction num/den of a turn
    // angle = 2 pi num / den
    if (8 * num <= den) return cx_cos_small(2 * kPi * num / den);
    if (4 * num <= den) return cx_sin_small(2 * kPi * (den - 4 * num) / (4.0 * den));      // cos(a) = sin(pi/2 - a)
    if (2 * num <= den) return -cx_cos_frac(den - 2 * num, 2 * den) ;                       // cos(a) = -cos(pi - a)
    return cx_cos_frac(den - num, den);                                                      // cos(a) = cos(2pi - a)
}
constexpr double cx_sin_frac(int num, int den) {
    // sin(a) = cos(a - pi/2) = cos(2 pi (num/den - 1/4)) = cos(2 pi (4 num - den) / (4 den))
    return cx_cos_frac(4 * num - den, 4 * den);
}
}  // namespace detail

template <int NUM, int DEN> struct Tw {
    static constexpr float c = (float)detail::cx_cos_frac(NUM, DEN);
    static constexpr float s = (float)detail::cx_sin_frac(NUM, DEN);
};

// complex values as register pairs; every helper below is one packed instruction
SNRX_HD float2 P(const cf& x) { return make_float2(x.r, x.i); }
SNRX_HD float2 Psw(const cf& x) { return make_float2(x.i, x.r); }          // swapped halves: folded into the operand
SNRX_HD cf C(const float2& x) { return cf{x.x, x.y}; }

// out0 = e + w*o ; out1 = e - w*o   with w = exp(+j 2 pi K / N)
template <int K, int N>
SNRX_HD void bfly(const cf& e, const cf& o, cf& out0, cf& out1) {
    constexpr int k = ((K % N) + N) % N;
    if constexpr (k == 0) {
        out0 = C(f2_add(P(e), P(o)));
        out1 = C(f2_fma(P(o), make_float2(-1.0f, -1.0f), P(e)));
    } else if constexpr (4 * k == N) {          // w = +j: w*o = (-o.i, o.r)
        out0 = C(f2_fma(Psw(o), make_float2(-1.0f, 1.0f), P(e)));
        out1 = C(f2_fma(Psw(o), make_float2(1.0f, -1.0f), P(e)));
    } else {
        constexpr float c = Tw<k, N>::c, s = Tw<k, N>::s;
        const float2 t = f2_fma(make_float2(-s, s), Psw(o), P(e));
        const float2 r0 = f2_fma(make_float2(c, c), P(o), t);
        out0 = C(r0);
        out1 = C(f2_fma(make_float2(2.0f, 2.0f), P(e), make_float2(-r0.x, -r0.y)));
    }
}

// N-point inverse DFT, N a power of two: in[0], in[S], in[2S], ... -> out[0..N-1] natural order
template <int N, int S>
struct IdftPow2 {
    SNRX_HD static void run(const cf* in, cf* out) {
        cf e[N / 2], o[N / 2];
        IdftPow2<N / 2, 2 * S>::run(in, e);
        IdftPow2<N / 2, 2 * S>::run(in + S, o);
        step<0>(e, o, out);
    }
    template <int K>
    SNRX_HD static void step(const cf* e, const cf* o, cf* out) {
        bfly<K, N>(e[K], o[K], out[K], out[K + N / 2]);
        if constexpr (K + 1 < N / 2) step<K + 1>(e, o, out);
    }
};
template <int S>
struct IdftPow2<1, S> {
    SNRX_HD static void run(const cf* in, cf* out) { out[0] = in[0]; }
};

// complex multiply by exp(+j 2 pi K / N)
template <int K, int N>
SNRX_HD cf twmul(const cf& x) {
    constexpr int k = ((K % N) + N) % N;
    if constexpr (k == 0) {
        return x;
    } else if constexpr (4 * k == N) {
        return cf{-x.i, x.r};
    } else if constexpr (2 * k == N) {
        return cf{-x.r, -x.i};
    } else if constexpr (4 * k == 3 * N) {
        return cf{x.i, -x.r};
    } else {
        constexpr float c = Tw<k, N>::c, s = Tw<k, N>::s;
        return C(f2_fma(make_float2(c, c), P(x), f2_mul(make_float2(-s, s), Psw(x))));
    }
}

// N = 3 * Q inverse DFT: r = 3*r2 + r1, k = k1 + Q*k2
//   Y[k1 + Q k2] = sum_{r1} W3^{k2 r1} * W_N^{k1 r1} * F_{r1}[k1],  F_{r1} = IDFT_Q(in[3 r2 + r1])
template <int N>
struct Idft3xQ {
    static constexpr int Q = N / 3;
    template <int K1>
    SNRX_HD static void combine(const cf* f0, const cf* f1, const cf* f2, cf* out) {
        constexpr float h = 0.86602540378443864676f;   // sqrt(3)/2
        const float2 a = P(f0[K1]);
        const cf bb = twmul<K1, N>(f1[K1]);
        const cf cc = twmul<2 * K1, N>(f2[K1]);
        const float2 s = f2_add(P(bb), P(cc));
        const float2 d = f2_fma(P(cc), make_float2(-1.0f, -1.0f), P(bb));
        out[K1] = C(f2_add(a, s));
        const float2 m = f2_fma(make_float2(-0.5f, -0.5f), s, a);
        // k2 = 1: a + w b + w^2 c, w = exp(+j 2pi/3) = -1/2 + j h  ->  m + j h d ;  k2 = 2: m - j h d
        const float2 dsw = make_float2(d.y, d.x);
        out[K1 + Q] = C(f2_fma(make_float2(-h, h), dsw, m));
        out[K1 + 2 * Q] = C(f2_fma(make_float2(h, -h), dsw, m));
        if constexpr (K1 + 1 < Q) combine<K1 + 1>(f0, f1, f2, out);
    }
    SNRX_HD static void run(const cf* in, cf* out) {
        cf f0[Q], f1[Q], f2[Q];
        IdftPow2<Q, 3>::run(in, f0);
        IdftPow2<Q, 3>::run(in + 1, f1);
        IdftPow2<Q, 3>::run(in + 2, f2);
        combine<0>(f0, f1, f2, out);
    }
};

// 48-point inverse DFT by the Good-Thomas prime-factor map, 48 = 3 * 16 with gcd(3, 16) = 1: no twiddles at all.
//   r = (16 n1 + 3 n2) mod 48,   k = (33 k16 + 16 k3) mod 48        (33 = 1 mod 16 = 0 mod 3;  16 = 0 mod 16 = 1 mod 3)
//   Y[k] = sum_{n1} W3^{k3 n1} F_{n1}[k16],   F_{n1}[k16] = sum_{n2} W16^{k16 n2} in[(16 n1 + 3 n2) mod 48]
// Pass n1 reads the same inputs as pass r1 = n1 of Idft3xQ<48> (r = 3 r2 + n1), in the order r2 = (5 n1 + n2) mod 16.
struct Pfa48 {
    SNRX_HD static constexpr int rot(int n1) { return 5 * n1 % 16; }                 // r2 of input n2 = 0 of pass n1
    SNRX_HD static constexpr int bin(int k16, int k3) { return (33 * k16 + 16 * k3) % 48; }
    template <int K16>
    SNRX_HD static void combine(const cf* f0, const cf* f1, const cf* f2, cf* out) {
        constexpr float h = 0.86602540378443864676f;   // sqrt(3)/2
        const float2 a = P(f0[K16]);
        const float2 s = f2_add(P(f1[K16]), P(f2[K16]));
        const float2 d = f2_fma(P(f2[K16]), make_float2(-1.0f, -1.0f), P(f1[K16]));
        out[bin(K16, 0)] = C(f2_add(a, s));
        const float2 m = f2_fma(make_float2(-0.5f, -0.5f), s, a);
        // k3 = 1: a + w b + w^2 c, w = exp(+j 2pi/3) = -1/2 + j h  ->  m + j h d ;  k3 = 2: m - j h d
        const float2 dsw = make_float2(d.y, d.x);
        out[bin(K16, 1)] = C(f2_fma(make_float2(-h, h), dsw, m));
        out[bin(K16, 2)] = C(f2_fma(make_float2(h, -h), dsw, m));
        if constexpr (K16 + 1 < 16) combine<K16 + 1>(f0, f1, f2, out);
    }
    SNRX_HD static void run(const cf* in, cf* out) {
        cf v[3][16], f[3][16];
        for (int n1 = 0; n1 < 3; n1++)
            for (int n2 = 0; n2 < 16; n2++) v[n1][n2] = in[(16 * n1 + 3 * n2) % 48];
        for (int n1 = 0; n1 < 3; n1++) IdftPow2<16, 1>::run(v[n1], f[n1]);
        combine<0>(f[0], f[1], f[2], out);
    }
};
constexpr bool pfa48_passes_agree() {
    for (int n1 = 0; n1 < 3; n1++)
        for (int n2 = 0; n2 < 16; n2++)
            if (3 * ((Pfa48::rot(n1) + n2) % 16) + n1 != (16 * n1 + 3 * n2) % 48) return false;
    return true;
}
static_assert(pfa48_passes_agree(), "pass n1 of the prime-factor map = the branches r = n1 (mod 3), rotated");

}  // namespace snrx
