// vsc_temporal.cuh — temporal depth stabilisation ahead of the frame pipeline (include/vsc_b200.h, vsc_submit_window).
//
// Frame t of a submission is filtered over the depth maps of its window (the frames t-k .. t+k the caller has).
// Two launches per submission:
//   temporal_sums_kernel    exact integer sums S_j, Q_j (every window plane) and P_tj (every frame / neighbour pair),
//                           one job per grid row, u64 integer atomics: the result does not depend on the order
//   temporal_filter_kernel  per frame a short prologue derives each neighbour's alignment (A, B) and the window that
//                           survives the cut rule in 128-bit integers and IEEE double, then every pixel takes the
//                           weighted mean of the aligned neighbours in f32 (weights from a shared-memory table)
// The f32 planes it writes enter the pipeline as VSC_DEPTH_F32 depth.  tests/temporal_oracle.py restates it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "vsc_common.cuh"

namespace vsc {

constexpr int TD_MAX_RADIUS = 8;
constexpr int TD_MAX_FRAMES = 4;                                          // frames of one submission
constexpr int TD_MAX_PLANES = TD_MAX_FRAMES + 2 * TD_MAX_RADIUS;         // window planes of one submission
constexpr int TD_MAX_PAIRS = TD_MAX_FRAMES * 2 * TD_MAX_RADIUS;
constexpr int TD_MAX_JOBS = TD_MAX_PLANES + TD_MAX_PAIRS;
constexpr int TD_SUMS = 2 * TD_MAX_PLANES + TD_MAX_PAIRS;                // u64 words of the sums buffer
constexpr double TD_MIN_R2 = 0.5;       // a neighbour whose squared correlation with D_t is below this is a scene cut
constexpr double TD_MAX_SLOPE = 16.0;   // ... and so is one that needs a larger alignment slope

struct TemporalArgs {
    const uint8_t* planes;      // window plane j at planes + j * stride
    long long stride;           // bytes, a multiple of 16
    long long npx;              // pixels per plane
    int np;                     // window planes
    int n;                      // frames filtered (window planes f0 .. f0 + n - 1)
    int f0;
    int k;                      // radius
    int maxv;                   // 255 or 65535
    // sums jobs: jb < 0: S and Q of plane ja; else P of the pair (ja = frame plane, jb = neighbour plane)
    signed char ja[TD_MAX_JOBS], jb[TD_MAX_JOBS];
    short jout[TD_MAX_JOBS];    // pair jobs: index into P
    unsigned long long* sums;   // S [np], Q [np], P [n * 2k]: pair (frame i, side s, distance m) at i*2k + s*k + m-1
    const float* wtab;          // w[m][d], [(k + 1) * 256]
    float* out[TD_MAX_FRAMES];  // f32 planes (room for npx rounded up to 4)
    int* win;                   // [2n]: lo, hi (window plane indices) per frame
};

// __int128 -> double, rounded to nearest, ties to even (Python's float(int)): the top 64 significant bits with a
// sticky bit for everything below them convert exactly as the whole number would.
__device__ __forceinline__ double td_i128_to_double(__int128 v) {
    const bool neg = v < 0;
    const unsigned __int128 m = neg ? (unsigned __int128)0 - (unsigned __int128)v : (unsigned __int128)v;
    const unsigned long long hi = (unsigned long long)(m >> 64);
    if (hi == 0) {
        const double r = __ull2double_rn((unsigned long long)m);
        return neg ? -r : r;
    }
    const int s = 64 - __clzll((long long)hi);                              // 1 .. 64 bits beyond the low word
    unsigned long long top = (unsigned long long)(m >> s);                  // bit 63 set
    top |= (unsigned long long)((m << (128 - s)) != 0);                     // sticky: below the rounding bit
    const double scale = __hiloint2double((1023 + s) << 20, 0);             // 2^s, exact
    const double r = __dmul_rn(__ull2double_rn(top), scale);
    return neg ? -r : r;
}

// Alignment of neighbour plane j to frame plane t (pair = index into P): false when the cut rule cuts it.
__device__ __forceinline__ bool td_align(const TemporalArgs& a, int t, int j, int pair, long long* A, long long* B) {
    const unsigned long long* S = a.sums;
    const unsigned long long* Q = a.sums + a.np;
    const unsigned long long* P = a.sums + 2 * a.np;
    const __int128 n = a.npx, st = S[t], sj = S[j];
    const __int128 cov = n * (__int128)P[pair] - st * sj;
    const __int128 vj = n * (__int128)Q[j] - sj * sj;
    const __int128 vt = n * (__int128)Q[t] - st * st;
    if (vj <= 0 || vt <= 0 || cov <= 0) return false;
    const double c = td_i128_to_double(cov), dvj = td_i128_to_double(vj), dvt = td_i128_to_double(vt);
    if (__dmul_rn(__dmul_rn(2.0, c), c) < __dmul_rn(dvj, dvt)) return false;          // r^2 < 1/2 (TD_MIN_R2)
    const double sl = __ddiv_rn(c, dvj);
    if (sl > TD_MAX_SLOPE) return false;
    const double b = __ddiv_rn(__dadd_rn(__ull2double_rn(S[t]), -__dmul_rn(sl, __ull2double_rn(S[j]))), (double)a.npx);
    *A = __double2ll_rn(__dmul_rn(sl, 65536.0));
    *B = __double2ll_rn(__dmul_rn(b, 65536.0));
    return true;
}

// per 32-bit word: sum, sum of squares, dot product of its elements
__device__ __forceinline__ void td_word(uint8_t, unsigned x, unsigned long long& s, unsigned long long& q) {
    s += __dp4a(x, 0x01010101u, 0u);
    q += __dp4a(x, x, 0u);
}
__device__ __forceinline__ void td_word(uint16_t, unsigned x, unsigned long long& s, unsigned long long& q) {
    const unsigned long long l = x & 0xffffu, h = x >> 16;
    s += l + h;
    q += l * l + h * h;
}
__device__ __forceinline__ unsigned long long td_dot(uint8_t, unsigned x, unsigned y) { return __dp4a(x, y, 0u); }
__device__ __forceinline__ unsigned long long td_dot(uint16_t, unsigned x, unsigned y) {
    return (unsigned long long)(x & 0xffffu) * (y & 0xffffu) + (unsigned long long)(x >> 16) * (y >> 16);
}

__device__ __forceinline__ unsigned long long td_warp_sum(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <typename T>
__global__ void __launch_bounds__(kThreads) temporal_sums_kernel(TemporalArgs a) {
    __shared__ unsigned long long red[2][kThreads / 32];
    const int job = blockIdx.y, pa = a.ja[job], pb = a.jb[job];
    const T* x = reinterpret_cast<const T*>(a.planes + pa * a.stride);
    const T* y = reinterpret_cast<const T*>(a.planes + (pb < 0 ? pa : pb) * a.stride);
    constexpr int V = 16 / sizeof(T);
    const long long nv = a.npx / V;
    unsigned long long s = 0, q = 0;
    const uint4* xv = reinterpret_cast<const uint4*>(x);
    const uint4* yv = reinterpret_cast<const uint4*>(y);
    if (pb < 0) {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
            const uint4 u = __ldg(xv + i);
            td_word(T(), u.x, s, q); td_word(T(), u.y, s, q); td_word(T(), u.z, s, q); td_word(T(), u.w, s, q);
        }
        if (blockIdx.x == 0)
            for (long long i = nv * V + threadIdx.x; i < a.npx; i += blockDim.x) {
                const unsigned long long v = x[i];
                s += v; q += v * v;
            }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
            const uint4 u = __ldg(xv + i), w = __ldg(yv + i);
            s += td_dot(T(), u.x, w.x) + td_dot(T(), u.y, w.y) + td_dot(T(), u.z, w.z) + td_dot(T(), u.w, w.w);
        }
        if (blockIdx.x == 0)
            for (long long i = nv * V + threadIdx.x; i < a.npx; i += blockDim.x) s += (unsigned long long)x[i] * y[i];
    }
    s = td_warp_sum(s);
    q = td_warp_sum(q);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { red[0][wid] = s; red[1][wid] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        s = 0; q = 0;
        for (int i = 0; i < kThreads / 32; i++) { s += red[0][i]; q += red[1][i]; }
        if (pb < 0) {
            atomicAdd(a.sums + pa, s);
            atomicAdd(a.sums + a.np + pa, q);
        } else {
            atomicAdd(a.sums + 2 * a.np + a.jout[job], s);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) temporal_filter_kernel(TemporalArgs a) {
    __shared__ float w_s[(TD_MAX_RADIUS + 1) * 256];
    __shared__ long long A_s[2 * TD_MAX_RADIUS], B_s[2 * TD_MAX_RADIUS];
    __shared__ int cut_s[2 * TD_MAX_RADIUS];
    __shared__ int lo_s, hi_s;
    const int i = blockIdx.y, t = a.f0 + i, k = a.k;
    for (int e = threadIdx.x; e < (k + 1) * 256; e += blockDim.x) w_s[e] = a.wtab[e];
    if (threadIdx.x < 2 * k) {                  // neighbour (side, m): thread side*k + m-1
        const int side = threadIdx.x / k, m = threadIdx.x % k + 1, j = side ? t + m : t - m;
        long long A = 0, B = 0;
        const bool ok = j >= 0 && j < a.np && td_align(a, t, j, i * 2 * k + threadIdx.x, &A, &B);
        cut_s[threadIdx.x] = !ok;
        A_s[threadIdx.x] = A;
        B_s[threadIdx.x] = B;
    }
    __syncthreads();
    if (threadIdx.x == 0) {                     // a cut also excludes everything farther out on its side
        int lo = t, hi = t;
        for (int m = 1; m <= k && !cut_s[m - 1]; m++) lo = t - m;
        for (int m = 1; m <= k && !cut_s[k + m - 1]; m++) hi = t + m;
        lo_s = lo; hi_s = hi;
        if (blockIdx.x == 0) { a.win[2 * i] = lo; a.win[2 * i + 1] = hi; }
    }
    __syncthreads();
    const int lo = lo_s, hi = hi_s, dshift = sizeof(T) == 2 ? 8 : 0;
    const long long nq = (a.npx + 3) / 4;
    float4* out = reinterpret_cast<float4*>(a.out[i]);
    for (long long qi = (long long)blockIdx.x * blockDim.x + threadIdx.x; qi < nq; qi += (long long)gridDim.x * blockDim.x) {
        int dt[4];
        {
            const T* p = reinterpret_cast<const T*>(a.planes + t * a.stride) + 4 * qi;
            if (sizeof(T) == 1) { const uchar4 v = *reinterpret_cast<const uchar4*>(p); dt[0] = v.x; dt[1] = v.y; dt[2] = v.z; dt[3] = v.w; }
            else { const ushort4 v = *reinterpret_cast<const ushort4*>(p); dt[0] = v.x; dt[1] = v.y; dt[2] = v.z; dt[3] = v.w; }
        }
        float num[4] = {0.f, 0.f, 0.f, 0.f}, den[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = lo; j <= hi; j++) {
            int e[4];
            const int m = j < t ? t - j : j - t;
            if (j == t) {
                e[0] = dt[0]; e[1] = dt[1]; e[2] = dt[2]; e[3] = dt[3];
            } else {
                const int nb = j < t ? m - 1 : k + m - 1;
                const long long A = A_s[nb], B = B_s[nb] + 32768;
                int dj[4];
                const T* p = reinterpret_cast<const T*>(a.planes + j * a.stride) + 4 * qi;
                if (sizeof(T) == 1) { const uchar4 v = *reinterpret_cast<const uchar4*>(p); dj[0] = v.x; dj[1] = v.y; dj[2] = v.z; dj[3] = v.w; }
                else { const ushort4 v = *reinterpret_cast<const ushort4*>(p); dj[0] = v.x; dj[1] = v.y; dj[2] = v.z; dj[3] = v.w; }
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const long long r = (A * dj[c] + B) >> 16;      // arithmetic shift: floor
                    e[c] = (int)(r < 0 ? 0 : (r > a.maxv ? a.maxv : r));
                }
            }
            const float* wm = w_s + m * 256;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                int d = (e[c] > dt[c] ? e[c] - dt[c] : dt[c] - e[c]) >> dshift;
                d = d < 255 ? d : 255;
                const float wt = wm[d];
                num[c] = __fadd_rn(num[c], __fmul_rn(wt, (float)e[c]));
                den[c] = __fadd_rn(den[c], wt);
            }
        }
        out[qi] = make_float4(__fdiv_rn(num[0], den[0]), __fdiv_rn(num[1], den[1]), __fdiv_rn(num[2], den[2]),
                              __fdiv_rn(num[3], den[3]));
    }
}

// test hook: n 128-bit two's-complement values (low word first) through td_i128_to_double
__global__ void temporal_convert_kernel(const unsigned long long* words, int n, double* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = td_i128_to_double((__int128)(((unsigned __int128)words[2 * i + 1] << 64) | words[2 * i]));
}

}  // namespace vsc
