// vsc_png.cuh — PNG encoding of the final rgb24 frame on the device (DESIGN.md section 2, "PNG output").
//
// The file is a fixed function of the frame (include/vsc_b200.h, VSC_ENCODE_PNG):
//   filter   every row gets the PNG filter (0..4) of least sum(min(b, 256 - b)) over its filtered bytes, ties to the
//            lowest type, row 0 filtered against a zero row (libpng's heuristic)           -> the filtered stream
//   deflate  the filtered stream cut into PNG_SEG-byte segments; each segment is one block parsed greedily into literals
//            and distance-1 matches of 3..258 bytes as zlib's Z_RLE does, with no match reaching before the segment.
//            The block is dynamic Huffman (lit/len code <= 15 bits, code-length code <= 7 bits, distance code: one
//            1-bit code for distance 1), or stored when that is not larger.  An empty stored block follows every
//            segment, so each segment ends byte-aligned and the segments concatenate as bytes.
//   framing  signature, IHDR, one IDAT per segment (the first also holds the zlib header 78 01, the last the final
//            empty fixed block 03 00 and the Adler-32), IEND.
// Three launches per submission, each covering every frame of the group: png_filter_kernel (one CTA per row),
// png_segment_kernel (one CTA per segment, the segment staged in shared memory) and png_assemble_kernel (one CTA per
// segment: offsets, chunk framing, Adler-32 combine, copy into the destination).  Every CRC-32 and the Adler-32 are
// computed here; the host only ever sees the finished file.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vsc {

constexpr int PNG_SEG = 32768;                                  // filtered-stream bytes per deflate segment (<= 65535)
constexpr int PNG_SEG_MAX = PNG_SEG + 10;                       // worst case: stored block (5 + n) + empty stored block
constexpr int PNG_SEG_STRIDE = (PNG_SEG_MAX + 255) / 256 * 256; // per-segment slot of the work buffer
constexpr int PNG_SEG_THREADS = 512;
constexpr int PNG_CHUNK = PNG_SEG / PNG_SEG_THREADS;            // segment bytes parsed by one thread
constexpr int PNG_MAX_FRAMES = 4;
constexpr int PNG_OUT_WORDS = (PNG_SEG_MAX + 3) / 4 + 2;
constexpr size_t PNG_SEG_SMEM = (size_t)PNG_SEG + (size_t)PNG_OUT_WORDS * 4;   // staged segment + packed block

struct PngSegMeta {
    uint32_t bytes;   // deflate bytes of the segment, sync-flush block included
    uint32_t crc;     // CRC-32 of "IDAT" (+ the zlib header for segment 0) + those bytes
    uint32_t a, b;    // the segment's Adler-32 sums: sum x_j and sum (n - j) x_j, mod 65521
};

struct PngArgs {
    const uint8_t* img[PNG_MAX_FRAMES];      // rgb24 frames [oh][ow][3] (device)
    uint8_t* filt[PNG_MAX_FRAMES];           // filtered stream, oh * (1 + 3 ow) bytes, 16-byte aligned
    uint8_t* seg[PNG_MAX_FRAMES];            // nseg * PNG_SEG_STRIDE deflate bytes
    PngSegMeta* meta[PNG_MAX_FRAMES];        // nseg entries
    uint8_t* dst[PNG_MAX_FRAMES];            // the file: device memory or page-locked host memory mapped into the device
    unsigned long long* size[PNG_MAX_FRAMES];   // file bytes
    unsigned long long* stats;               // null, or 3 counters: lit/len codes length-limited, code-length codes
                                             // length-limited, stored segments
    int oh, ow, nseg;
    long long n;                             // filtered-stream bytes
};

// x^(2^k) mod the CRC-32 polynomial (reflected), k = 0..31: zlib's x2n_table
__constant__ uint32_t c_png_x2n[32] = {
    0x40000000, 0x20000000, 0x08000000, 0x00800000, 0x00008000, 0xedb88320, 0xb1e6b092, 0xa06a2517, 0xed627dae, 0x88d14467,
    0xd7bbfe6a, 0xec447f11, 0x8e7ea170, 0x6427800e, 0x4d47bae0, 0x09fe548f, 0x83852d0f, 0x30362f1a, 0x7b5a9cc3, 0x31fec169,
    0x9fec022a, 0x6c8dedc4, 0x15d6874d, 0x5fde7a4e, 0xbad90e37, 0x2e4e5eef, 0x4eaba214, 0xa8a472c0, 0x429a969e, 0x148d302a,
    0xc40ba6d0, 0xc4e22c3c};
__constant__ uint16_t c_png_len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83,
                                            99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_png_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint8_t c_png_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__device__ __forceinline__ uint32_t png_multmodp(uint32_t a, uint32_t b) {   // a * b mod P (reflected), zlib's multmodp
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// crc32(A || B) from crc32(A), crc32(B) and |B|
__device__ __forceinline__ uint32_t png_crc_combine(uint32_t c1, uint32_t c2, uint32_t len2) {
    uint32_t p = 1u << 31;
    for (int k = 3; len2; len2 >>= 1, k++)
        if (len2 & 1) p = png_multmodp(c_png_x2n[k & 31], p);
    return png_multmodp(p, c1) ^ c2;
}
__device__ __forceinline__ uint32_t png_crc_bytes(uint32_t crc, const uint8_t* p, int n) {   // bitwise, for a few bytes
    uint32_t c = ~crc;
    for (int i = 0; i < n; i++) {
        c ^= p[i];
        for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
    }
    return ~c;
}
__device__ __forceinline__ void png_be32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// ---- filter ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int png_cost(int v) { v &= 255; return v < 128 ? v : 256 - v; }
__device__ __forceinline__ int png_paeth(int a, int b, int c) {
    const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}
__device__ __forceinline__ int png_filtered(int type, int x, int l, int u, int ul) {
    switch (type) {
        case 0: return x;
        case 1: return x - l;
        case 2: return x - u;
        case 3: return x - ((l + u) >> 1);
        default: return x - png_paeth(l, u, ul);
    }
}

// grid (oh, frames), 256 threads: one row per CTA
__global__ void __launch_bounds__(256) png_filter_kernel(PngArgs a) {
    const int y = blockIdx.x, f = blockIdx.y, rb = 3 * a.ow;
    const uint8_t* cur = a.img[f] + (size_t)y * rb;
    const uint8_t* up = cur - rb;
    uint8_t* out = a.filt[f] + (size_t)y * (rb + 1);
    unsigned c[5] = {0, 0, 0, 0, 0};
    for (int i = threadIdx.x; i < rb; i += blockDim.x) {
        const int x = cur[i], l = i >= 3 ? cur[i - 3] : 0, u = y ? up[i] : 0, ul = (y && i >= 3) ? up[i - 3] : 0;
#pragma unroll
        for (int t = 0; t < 5; t++) c[t] += png_cost(png_filtered(t, x, l, u, ul));
    }
    __shared__ unsigned red[8][5];
    __shared__ int type;
#pragma unroll
    for (int t = 0; t < 5; t++) {
        unsigned v = c[t];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][t] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned best = 0xffffffffu;
        int bt = 0;
        for (int t = 0; t < 5; t++) {
            unsigned s = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w][t];
            if (s < best) { best = s; bt = t; }
        }
        type = bt;
        out[0] = (uint8_t)bt;
    }
    __syncthreads();
    const int bt = type;
    for (int i = threadIdx.x; i < rb; i += blockDim.x) {
        const int x = cur[i], l = i >= 3 ? cur[i - 3] : 0, u = y ? up[i] : 0, ul = (y && i >= 3) ? up[i - 3] : 0;
        out[1 + i] = (uint8_t)png_filtered(bt, x, l, u, ul);
    }
}

// ---- segment ------------------------------------------------------------------------------------------------------
struct PngSegShared {
    unsigned hist[288];          // lit/len frequencies; then the code-length frequencies in [0, 19)
    uint16_t code[288];          // bit-reversed canonical codes
    uint8_t len[288];
    uint16_t cl_code[19];
    uint8_t cl_len[19];
    uint8_t len_code[259];       // match length -> length code index (0..28)
    uint8_t rle_sym[320], rle_ext[320];
    int n_rle, hlit, hclen;
    uint32_t crc_tab[256];
    // Huffman construction
    unsigned w[576];
    uint16_t par[576], dep[576], sorted[288];
    unsigned cnt[16], next[16];
    int m, limited;
    // block scans
    unsigned long long scan[PNG_SEG_THREADS];
    uint32_t crc[PNG_SEG_THREADS], clen[PNG_SEG_THREADS];
    unsigned hdr_bits, body_bits;
};

// exclusive scan over the block's threads in order (reverse: from the last thread down); *total = the whole reduction
template <typename T, typename Op>
__device__ __forceinline__ T png_block_scan(T v, T id, Op op, T* buf, bool reverse, T* total) {
    const int n = blockDim.x, t = reverse ? n - 1 - threadIdx.x : threadIdx.x;
    buf[t] = v;
    __syncthreads();
    for (int off = 1; off < n; off <<= 1) {
        const T x = t >= off ? buf[t - off] : id;
        __syncthreads();
        buf[t] = op(buf[t], x);
        __syncthreads();
    }
    const T r = t ? buf[t - 1] : id;
    if (total) *total = buf[n - 1];
    __syncthreads();
    return r;
}

// Code lengths of a Huffman code for freq[0, nsym) limited to maxlen bits (whole block).  Leaves are ranked by
// (frequency, symbol); the tree is built from two queues; over-long leaves are clamped and the Kraft sum repaired as
// miniz does (one code at maxlen dropped, one shorter code split, until the code is complete); lengths then go to the
// symbols in rank order, shortest to the most frequent.  A single used symbol gets length 1.  Returns 1 if the limit
// had to be enforced.
__device__ int png_huffman(const unsigned* freq, int nsym, int maxlen, uint8_t* len, PngSegShared& S) {
    if (threadIdx.x == 0) S.m = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < nsym; i += blockDim.x) {
        len[i] = 0;
        const unsigned fi = freq[i];
        if (fi) {
            int r = 0;
            for (int j = 0; j < nsym; j++) {
                const unsigned fj = freq[j];
                r += fj && (fj < fi || (fj == fi && j < i));
            }
            S.sorted[r] = (uint16_t)i;
            atomicAdd(&S.m, 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int m = S.m;
        int limited = 0;
        if (m == 1) {
            len[S.sorted[0]] = 1;
        } else if (m > 1) {
            for (int i = 0; i < m; i++) S.w[i] = freq[S.sorted[i]];
            int li = 0, ii = m;
            for (int nx = m; nx < 2 * m - 1; nx++) {
                const int p0 = (li < m && (ii >= nx || S.w[li] <= S.w[ii])) ? li++ : ii++;
                const int p1 = (li < m && (ii >= nx || S.w[li] <= S.w[ii])) ? li++ : ii++;
                S.w[nx] = S.w[p0] + S.w[p1];
                S.par[p0] = (uint16_t)nx;
                S.par[p1] = (uint16_t)nx;
            }
            for (int b = 0; b < 16; b++) S.cnt[b] = 0;
            S.dep[2 * m - 2] = 0;
            for (int i = 2 * m - 3; i >= 0; i--) {
                S.dep[i] = S.dep[S.par[i]] + 1;
                if (i < m) {
                    int d = S.dep[i];
                    if (d > maxlen) { d = maxlen; limited = 1; }
                    S.cnt[d]++;
                }
            }
            if (limited) {
                unsigned total = 0;
                for (int b = maxlen; b > 0; b--) total += S.cnt[b] << (maxlen - b);
                while (total != (1u << maxlen)) {
                    S.cnt[maxlen]--;
                    for (int b = maxlen - 1; b > 0; b--)
                        if (S.cnt[b]) { S.cnt[b]--; S.cnt[b + 1] += 2; break; }
                    total--;
                }
            }
            int j = m;
            for (int b = 1; b <= maxlen; b++)
                for (unsigned c = S.cnt[b]; c; c--) len[S.sorted[--j]] = (uint8_t)b;
        }
        S.limited = limited;
    }
    __syncthreads();
    return S.limited;
}
// canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first packing; one thread
__device__ void png_canonical(const uint8_t* len, int n, uint16_t* code, PngSegShared& S) {
    for (int b = 0; b < 16; b++) S.cnt[b] = 0;
    for (int i = 0; i < n; i++) S.cnt[len[i]]++;
    S.cnt[0] = 0;
    unsigned c = 0;
    for (int b = 1; b < 16; b++) { c = (c + S.cnt[b - 1]) << 1; S.next[b] = c; }
    for (int i = 0; i < n; i++)
        if (len[i]) code[i] = (uint16_t)(__brev(S.next[len[i]]++) >> (32 - len[i]));
}

__device__ __forceinline__ void png_put(uint32_t* w, unsigned pos, uint32_t bits, int nbits) {
    if (!nbits) return;
    const unsigned sh = pos & 31;
    atomicOr(&w[pos >> 5], bits << sh);
    if (sh + nbits > 32) atomicOr(&w[(pos >> 5) + 1], bits >> (32 - sh));
}

// The Z_RLE parse of bytes [cs, ce) of a segment of n bytes: a maximal run of length L is one literal, then
// (L - 1) / 258 matches of 258, then the rest as one match if it has >= 3 bytes, else as literals.  carry_s is the
// start of the run holding cs, carry_e the end of the run holding ce (both only read when the run crosses the edge).
// f.lit(byte) / f.match(length) in stream order.
template <typename F>
__device__ __forceinline__ void png_symbols(const uint8_t* in, int cs, int ce, int n, int carry_s, int carry_e, F& f) {
    int s = carry_s, e = 0;
    bool have_e = false;
    for (int i = cs; i < ce; i++) {
        const int v = in[i];
        if (i == 0 || in[i - 1] != v) { s = i; have_e = false; }
        if (!have_e) {
            int j = i + 1;
            while (j < ce && in[j] == v) j++;
            e = (j == ce && j < n && in[j] == v) ? carry_e : j;
            have_e = true;
        }
        const int off = i - s;
        if (off == 0) { f.lit(v); continue; }
        const int T = e - s - 1, t = off - 1, k = T / 258, r = T - 258 * k;
        if (t < 258 * k) {
            const int q = t % 258;
            if (q == 0) { f.match(258); i += 257; }
            else i += 257 - q;                   // inside a match that started in an earlier chunk
        } else if (r >= 3) {
            if (t == 258 * k) f.match(r);
            i = e - 1;
        } else {
            f.lit(v);
        }
    }
}

struct PngHist {
    PngSegShared& S;
    __device__ void lit(int v) { atomicAdd(&S.hist[v], 1u); }
    __device__ void match(int L) { atomicAdd(&S.hist[257 + S.len_code[L]], 1u); }
};
struct PngBits {
    const PngSegShared& S;
    unsigned bits;
    __device__ void lit(int v) { bits += S.len[v]; }
    __device__ void match(int L) { const int c = S.len_code[L]; bits += S.len[257 + c] + c_png_len_extra[c] + 1; }
};
struct PngPack {
    const PngSegShared& S;
    uint32_t* w;
    unsigned pos;
    __device__ void lit(int v) { png_put(w, pos, S.code[v], S.len[v]); pos += S.len[v]; }
    __device__ void match(int L) {
        const int c = S.len_code[L], l = S.len[257 + c], x = c_png_len_extra[c];
        png_put(w, pos, S.code[257 + c] | ((uint32_t)(L - c_png_len_base[c]) << l), l + x);
        pos += l + x + 1;                        // + the 1-bit code 0 of distance 1
    }
};

// grid (nseg, frames), PNG_SEG_THREADS threads, PNG_SEG_SMEM bytes of dynamic shared memory
__global__ void __launch_bounds__(PNG_SEG_THREADS) png_segment_kernel(PngArgs a) {
    extern __shared__ __align__(16) uint8_t png_dyn[];
    __shared__ PngSegShared S;
    uint8_t* in = png_dyn;
    uint32_t* ow = reinterpret_cast<uint32_t*>(png_dyn + PNG_SEG);
    uint8_t* ob = reinterpret_cast<uint8_t*>(ow);
    const int k = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
    const long long o = (long long)k * PNG_SEG;
    const int n = (int)min((long long)PNG_SEG, a.n - o);

    // stage the segment (16-byte loads: segment starts are 16-byte aligned) and the tables
    const uint8_t* src = a.filt[f] + o;
    for (int i = tid; i < n / 16; i += nt) reinterpret_cast<uint4*>(in)[i] = reinterpret_cast<const uint4*>(src)[i];
    for (int i = n / 16 * 16 + tid; i < n; i += nt) in[i] = src[i];
    for (int i = tid; i < 256; i += nt) {
        uint32_t c = i;
        for (int b = 0; b < 8; b++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
        S.crc_tab[i] = c;
    }
    for (int i = tid; i < 288; i += nt) S.hist[i] = i == 256;    // end of block
    for (int L = 3 + tid; L <= 258; L += nt) {
        int c = 28;
        while (c_png_len_base[c] > L) c--;
        S.len_code[L] = (uint8_t)c;
    }
    __syncthreads();

    // Adler-32 sums and run edges of this thread's chunk
    const int cs = min(tid * PNG_CHUNK, n), ce = min(cs + PNG_CHUNK, n);
    unsigned long long sa = 0, sb = 0;
    int last_start = -1, first_end = n;
    for (int i = cs; i < ce; i++) {
        const unsigned x = in[i];
        sa += x;
        sb += (unsigned long long)x * (unsigned)(n - i);
        if (i == 0 || in[i - 1] != in[i]) last_start = i;
        if (first_end == n && (i == n - 1 || in[i] != in[i + 1])) first_end = i + 1;
    }
    unsigned long long ta, tb;
    png_block_scan<unsigned long long>(sa, 0ull, [](unsigned long long x, unsigned long long y) { return x + y; }, S.scan, false, &ta);
    png_block_scan<unsigned long long>(sb, 0ull, [](unsigned long long x, unsigned long long y) { return x + y; }, S.scan, false, &tb);
    const int carry_s = (int)(long long)png_block_scan<unsigned long long>(
        (unsigned long long)(last_start + 1), 0ull, [](unsigned long long x, unsigned long long y) { return x > y ? x : y; },
        S.scan, false, nullptr) - 1;
    const int carry_e = (int)png_block_scan<unsigned long long>(
        (unsigned long long)first_end, (unsigned long long)n, [](unsigned long long x, unsigned long long y) { return x < y ? x : y; },
        S.scan, true, nullptr);

    // histogram, then the lit/len code
    {
        PngHist h{S};
        png_symbols(in, cs, ce, n, carry_s, carry_e, h);
    }
    __syncthreads();
    const int lim_ll = png_huffman(S.hist, 286, 15, S.len, S);
    if (tid == 0) {
        png_canonical(S.len, 286, S.code, S);
        // lit/len lengths + the one distance length, run-length coded with 16 / 17 / 18
        int hlit = 286;
        while (hlit > 257 && S.len[hlit - 1] == 0) hlit--;
        S.hlit = hlit;
        const int tot = hlit + 1;
        int nr = 0;
        for (int i = 0; i < 19; i++) S.hist[i] = 0;
        for (int i = 0; i < tot;) {
            const int v = i < hlit ? S.len[i] : 1;
            int r = 1;
            while (i + r < tot && (i + r < hlit ? S.len[i + r] : 1) == v) r++;
            i += r;
            if (v == 0) {
                while (r >= 11) { const int q = min(r, 138); S.rle_sym[nr] = 18; S.rle_ext[nr++] = (uint8_t)(q - 11); r -= q; }
                if (r >= 3) { S.rle_sym[nr] = 17; S.rle_ext[nr++] = (uint8_t)(r - 3); r = 0; }
            } else {
                S.rle_sym[nr] = (uint8_t)v; S.rle_ext[nr++] = 0; r--;
                while (r >= 3) { const int q = min(r, 6); S.rle_sym[nr] = 16; S.rle_ext[nr++] = (uint8_t)(q - 3); r -= q; }
            }
            for (; r > 0; r--) { S.rle_sym[nr] = (uint8_t)v; S.rle_ext[nr++] = 0; }
        }
        S.n_rle = nr;
        for (int i = 0; i < nr; i++) S.hist[S.rle_sym[i]]++;
    }
    __syncthreads();
    const int lim_cl = png_huffman(S.hist, 19, 7, S.cl_len, S);
    if (tid == 0) {
        png_canonical(S.cl_len, 19, S.cl_code, S);
        int hclen = 19;
        while (hclen > 4 && S.cl_len[c_png_cl_order[hclen - 1]] == 0) hclen--;
        S.hclen = hclen;
        unsigned bits = 3 + 14 + 3 * hclen;
        for (int i = 0; i < S.n_rle; i++) {
            const int sy = S.rle_sym[i];
            bits += S.cl_len[sy] + (sy == 16 ? 2 : sy == 17 ? 3 : sy == 18 ? 7 : 0);
        }
        S.hdr_bits = bits;
    }
    PngBits pb{S, 0};
    png_symbols(in, cs, ce, n, carry_s, carry_e, pb);
    unsigned body;
    const unsigned boff = (unsigned)png_block_scan<unsigned long long>(
        pb.bits, 0ull, [](unsigned long long x, unsigned long long y) { return x + y; }, S.scan, false, nullptr);
    if (tid == nt - 1) S.body_bits = boff + pb.bits;
    __syncthreads();
    body = S.body_bits;
    const unsigned dyn_bits = S.hdr_bits + body + S.len[256];
    const int dyn_bytes = (int)((dyn_bits + 3 + 7) / 8) + 4;
    const bool stored = dyn_bytes >= n + 10;
    const int D = stored ? n + 10 : dyn_bytes;

    if (!stored) {
        for (int i = tid; i < (D + 3) / 4; i += nt) ow[i] = 0;
        __syncthreads();
        if (tid == 0) {
            unsigned p = 0;
            png_put(ow, p, 4u, 3); p += 3;                       // BFINAL 0, BTYPE 10
            png_put(ow, p, (uint32_t)(S.hlit - 257), 5); p += 5;
            p += 5;                                              // HDIST - 1 = 0
            png_put(ow, p, (uint32_t)(S.hclen - 4), 4); p += 4;
            for (int i = 0; i < S.hclen; i++) { png_put(ow, p, S.cl_len[c_png_cl_order[i]], 3); p += 3; }
            for (int i = 0; i < S.n_rle; i++) {
                const int sy = S.rle_sym[i], x = sy == 16 ? 2 : sy == 17 ? 3 : sy == 18 ? 7 : 0;
                png_put(ow, p, S.cl_code[sy] | ((uint32_t)S.rle_ext[i] << S.cl_len[sy]), S.cl_len[sy] + x);
                p += S.cl_len[sy] + x;
            }
            const unsigned pe = S.hdr_bits + body;
            png_put(ow, pe, S.code[256], S.len[256]);            // end of block
        }
        PngPack pk{S, ow, S.hdr_bits + boff};
        png_symbols(in, cs, ce, n, carry_s, carry_e, pk);
        __syncthreads();
        // the empty stored block: 3 zero bits, padding, LEN 00 00 (already zero), NLEN FF FF
        if (tid == 0) { ob[D - 2] = 0xff; ob[D - 1] = 0xff; }
    } else {
        for (int i = tid; i < n; i += nt) ob[5 + i] = in[i];
        if (tid == 0) {
            ob[0] = 0; ob[1] = (uint8_t)n; ob[2] = (uint8_t)(n >> 8); ob[3] = (uint8_t)~n; ob[4] = (uint8_t)(~n >> 8);
            ob[5 + n] = 0; ob[6 + n] = 0; ob[7 + n] = 0; ob[8 + n] = 0xff; ob[9 + n] = 0xff;
        }
    }
    __syncthreads();

    // CRC-32 of the chunk's bytes so far: per-thread pieces combined in a tree
    const int per = (D + nt - 1) / nt, ps = min(tid * per, D), pe = min(ps + per, D);
    uint32_t c = 0xffffffffu;
    for (int i = ps; i < pe; i++) c = S.crc_tab[(c ^ ob[i]) & 255] ^ (c >> 8);
    S.crc[tid] = ~c;
    S.clen[tid] = (uint32_t)(pe - ps);
    __syncthreads();
    for (int st = 1; st < nt; st <<= 1) {
        if ((tid & (2 * st - 1)) == 0 && tid + st < nt) {
            S.crc[tid] = png_crc_combine(S.crc[tid], S.crc[tid + st], S.clen[tid + st]);
            S.clen[tid] += S.clen[tid + st];
        }
        __syncthreads();
    }
    uint8_t* dst = a.seg[f] + (size_t)k * PNG_SEG_STRIDE;
    for (int i = tid; i < (D + 3) / 4; i += nt) reinterpret_cast<uint32_t*>(dst)[i] = ow[i];
    if (tid == 0) {
        const uint8_t pre[6] = {'I', 'D', 'A', 'T', 0x78, 0x01};
        const uint32_t cp = png_crc_bytes(0, pre, k == 0 ? 6 : 4);
        PngSegMeta mt;
        mt.bytes = (uint32_t)D;
        mt.crc = png_crc_combine(cp, S.crc[0], (uint32_t)D);
        mt.a = (uint32_t)(ta % 65521u);
        mt.b = (uint32_t)(tb % 65521u);
        a.meta[f][k] = mt;
        if (a.stats) {
            if (lim_ll) atomicAdd(&a.stats[0], 1ull);
            if (lim_cl) atomicAdd(&a.stats[1], 1ull);
            if (stored) atomicAdd(&a.stats[2], 1ull);
        }
    }
}

// ---- assemble -----------------------------------------------------------------------------------------------------
// grid (nseg, frames), 256 threads: CTA k writes IDAT chunk k at its offset (CTA 0 also the signature and IHDR, the last
// CTA the final block, the Adler-32, IEND and the file size)
__global__ void __launch_bounds__(256) png_assemble_kernel(PngArgs a) {
    const int k = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
    const PngSegMeta* meta = a.meta[f];
    const bool last = k == a.nseg - 1;
    __shared__ unsigned long long red[3][256];
    unsigned long long s = 0, sa = 0, sb = 0;
    for (int j = tid; j < k; j += nt) s += meta[j].bytes;
    if (last) {
        const unsigned long long N = (unsigned long long)a.n;
        for (int j = tid; j < a.nseg; j += nt) {
            const unsigned long long after = N - min(N, (unsigned long long)(j + 1) * PNG_SEG);
            sa += meta[j].a;
            sb += (meta[j].b + (unsigned long long)meta[j].a * (after % 65521u)) % 65521u;
        }
    }
    red[0][tid] = s; red[1][tid] = sa; red[2][tid] = sb;
    __syncthreads();
    for (int st = nt / 2; st; st >>= 1) {
        if (tid < st) for (int q = 0; q < 3; q++) red[q][tid] += red[q][tid + st];
        __syncthreads();
    }
    const PngSegMeta mk = meta[k];
    const size_t off = 33 + 12 * (size_t)k + (k > 0 ? 2 : 0) + red[0][0];   // chunk k
    const int head = k == 0 ? 2 : 0;
    const uint32_t dlen = mk.bytes + head + (last ? 6 : 0);
    uint8_t* o = a.dst[f] + off;
    const uint8_t* src = a.seg[f] + (size_t)k * PNG_SEG_STRIDE;
    for (uint32_t i = tid; i < mk.bytes; i += nt) o[8 + head + i] = src[i];
    if (tid == 0) {
        png_be32(o, dlen);
        o[4] = 'I'; o[5] = 'D'; o[6] = 'A'; o[7] = 'T';
        if (k == 0) { o[8] = 0x78; o[9] = 0x01; }
        uint32_t crc = mk.crc;
        uint8_t* t = o + 8 + head + mk.bytes;
        if (last) {
            const uint32_t ad_a = (uint32_t)((1 + red[1][0]) % 65521u);
            const uint32_t ad_b = (uint32_t)(((unsigned long long)a.n % 65521u + red[2][0]) % 65521u);
            uint8_t tail[6] = {0x03, 0x00};
            png_be32(tail + 2, ad_b << 16 | ad_a);
            for (int i = 0; i < 6; i++) t[i] = tail[i];
            crc = png_crc_bytes(crc, tail, 6);
            t += 6;
            png_be32(t, crc);
            const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
            for (int i = 0; i < 12; i++) t[4 + i] = iend[i];
            *a.size[f] = (unsigned long long)(off + 12 + dlen + 12);
        } else {
            png_be32(t, crc);
        }
        if (k == 0) {
            uint8_t* h = a.dst[f];
            const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
            uint8_t ihdr[17] = {'I', 'H', 'D', 'R'};
            png_be32(ihdr + 4, (uint32_t)a.ow);
            png_be32(ihdr + 8, (uint32_t)a.oh);
            ihdr[12] = 8; ihdr[13] = 2; ihdr[14] = 0; ihdr[15] = 0; ihdr[16] = 0;
            for (int i = 0; i < 8; i++) h[i] = sig[i];
            png_be32(h + 8, 13);
            for (int i = 0; i < 17; i++) h[12 + i] = ihdr[i];
            png_be32(h + 29, png_crc_bytes(0, ihdr, 17));
        }
    }
}

}  // namespace vsc
