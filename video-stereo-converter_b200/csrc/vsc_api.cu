// vsc_api.cu — host side of libvsc_b200.so: the C ABI declared in include/vsc_b200.h.
//
// One vsc_ctx owns `n_slots` frame slots.  A slot is everything one in-flight frame needs:
// a CUDA stream, device buffers (grown on demand, never shrunk), the host-computed tap tables for
// its geometry and a pinned mirror of the per-frame scalars.  Frames submitted to different slots
// overlap (H2D copy / kernels / D2H copy of neighbouring frames run concurrently on the copy
// engines and SMs); there is no cross-frame state, mirroring the reference where process_frame is
// a pure function of (rgb, depth, params) (stereo_core.py:225-311).
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/vsc_b200.h"
#include "vsc_march.cuh"
#include "vsc_png.cuh"

using namespace vsc;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(VSC_E_CUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__, \
                        cudaGetErrorString(e_));                                                   \
    } while (0)

// ------------------------------------------------------------------------------------------------
// host tables (all float math below follows the oracle / the libraries bit for bit; this file is
// compiled with -ffp-contract=off)
// ------------------------------------------------------------------------------------------------
static void lanczos4_coeffs(float x, float* c) {   // OpenCV interpolateLanczos4
    static const double s45 = 0.70710678118654752440084436210485;
    static const double cs[8][2] = {{1, 0}, {-s45, -s45}, {0, 1}, {s45, -s45}, {-1, 0}, {s45, s45}, {0, -1}, {-s45, s45}};
    const double PI = 3.1415926535897932384626433832795;
    float sum = 0.f;
    double y0 = -(x + 3) * PI * 0.25, s0 = sin(y0), c0 = cos(y0);
    for (int i = 0; i < 8; i++) {
        float y0_ = (x + 3 - i);
        if (fabsf(y0_) >= 1e-6f) {
            double y = -y0_ * PI * 0.25;
            c[i] = (float)((cs[i][0] * s0 + cs[i][1] * c0) / (y * y));
        } else {
            c[i] = 1e30f;
        }
        sum += c[i];
    }
    sum = 1.f / sum;
    for (int i = 0; i < 8; i++) c[i] *= sum;
}
static short sat_short(float v) {
    long r = lrintf(v);
    return (short)(r < -32768 ? -32768 : (r > 32767 ? 32767 : r));
}
static void lanczos_tables(int W, int dW, std::vector<int>& sx0, std::vector<float>& ft, std::vector<short>& it) {
    sx0.resize(dW); ft.resize(8 * (size_t)dW); it.resize(8 * (size_t)dW);
    const double inv_scale = (double)dW / (double)W, scale = 1.0 / inv_scale;
    for (int dx = 0; dx < dW; dx++) {
        float fx = (float)((dx + 0.5) * scale - 0.5);
        int sx = (int)floorf(fx);
        fx -= (float)sx;
        sx0[dx] = sx - 3;
        lanczos4_coeffs(fx, &ft[8 * (size_t)dx]);
        for (int k = 0; k < 8; k++) it[8 * (size_t)dx + k] = sat_short(ft[8 * (size_t)dx + k] * 2048.f);
    }
}
static void axis_table(int in, int out, std::vector<AxisTap>& t) {   // ATen bilinear source index / lambda
    t.resize(out);
    const float scale = (float)in / (float)out;
    for (int o = 0; o < out; o++) {
        float s = fmaf(scale, (float)o + 0.5f, -0.5f);
        if (s < 0.f) s = 0.f;
        int a = (int)floorf(s);
        if (a > in - 1) a = in - 1;
        float lam = s - (float)a;
        lam = lam < 0.f ? 0.f : (lam > 1.f ? 1.f : lam);
        t[o].i0 = a;
        t[o].i1 = a + 1 < in ? a + 1 : in - 1;
        t[o].l1 = lam;
        t[o].l0 = 1.f - lam;
    }
}
// torch.sum of a short f32 vector in ATen's CPU order (see oracle.py:_torch_sum_f32)
static float torch_sum_f32(const float* x, int n) {
    if (n < 8) {
        float acc[4] = {0, 0, 0, 0};
        int nb = n / 4;
        for (int b = 0; b < nb; b++) for (int k = 0; k < 4; k++) acc[k] = acc[k] + x[b * 4 + k];
        for (int i = nb * 4; i < n; i++) acc[0] = acc[0] + x[i];
        for (int k = 1; k < 4; k++) acc[0] = acc[0] + acc[k];
        return acc[0];
    }
    float acc[4][8];
    memset(acc, 0, sizeof acc);
    int vs = n / 8, nb = vs / 4;
    for (int b = 0; b < nb; b++) for (int k = 0; k < 4; k++) for (int l = 0; l < 8; l++) acc[k][l] += x[(b * 4 + k) * 8 + l];
    for (int i = nb * 4; i < vs; i++) for (int l = 0; l < 8; l++) acc[0][l] += x[i * 8 + l];
    for (int k = 1; k < 4; k++) for (int l = 0; l < 8; l++) acc[0][l] += acc[k][l];
    float s = 0.f;
    for (int i = vs * 8; i < n; i++) s += x[i];
    for (int l = 0; l < 8; l++) s += acc[0][l];
    return s;
}
static GaussTaps gauss_taps(int k, double sigma) {   // kornia get_gaussian_kernel1d, f32
    GaussTaps t;
    memset(&t, 0, sizeof t);
    t.k = k;
    if (k <= 0) return t;
    const float den = (float)(2.0 * sigma * sigma);
    float g[31];
    for (int i = 0; i < k; i++) {
        float n = (float)i - (float)(k / 2);
        float arg = -(n * n) / den;
        g[i] = (float)exp((double)arg);
    }
    const float s = torch_sum_f32(g, k);
    for (int i = 0; i < k; i++) t.g[i] = g[i] / s;
    return t;
}
static void bilateral_tables(int d, double sigma_color, double sigma_space, float* color_w, BilateralTaps& bt) {
    if (sigma_color <= 0) sigma_color = 1;
    if (sigma_space <= 0) sigma_space = 1;
    const double gc = -0.5 / (sigma_color * sigma_color), gs = -0.5 / (sigma_space * sigma_space);
    int radius = d <= 0 ? (int)lrint(sigma_space * 1.5) : d / 2;
    if (radius < 1) radius = 1;
    if (color_w) for (int i = 0; i < 768; i++) color_w[i] = (float)exp((double)i * i * gc);
    bt.n = 0; bt.radius = radius;
    for (int i = -radius; i <= radius; i++)
        for (int j = -radius; j <= radius; j++) {
            double r = sqrt((double)i * i + (double)j * j);
            if (r > radius) continue;
            bt.w[bt.n] = (float)exp(r * r * gs);
            bt.dy[bt.n] = (signed char)i; bt.dx[bt.n] = (signed char)j;
            bt.n++;
        }
}

// ------------------------------------------------------------------------------------------------
// geometry (stereo_core.py:249-251, 275-289, 364-365, 384, 409)
// ------------------------------------------------------------------------------------------------
extern "C" int vsc_abi_version(void) { return VSC_ABI_VERSION; }
extern "C" const char* vsc_last_error(void) { return g_err.c_str(); }
extern "C" void vsc_default_params(vsc_params* p) {
    p->max_disparity = 50.0; p->convergence = -10.0; p->super_sampling = 3.0; p->edge_softness = 20.0;
    p->artifact_smoothing = 1.0; p->depth_gamma = 0.2; p->sharpen = 14.0;
}
extern "C" int vsc_geometry(int H, int W, const vsc_params* p, vsc_geom* g) {
    if (!p || !g) return fail(VSC_E_INVALID, "null argument");
    if (H < 8 || W < 8) return fail(VSC_E_INVALID, "frame %dx%d is smaller than 8x8", W, H);
    if (!(p->max_disparity >= 0) || !(p->super_sampling > 0) || !(p->depth_gamma > 0) || !(p->edge_softness >= 0) ||
        !(p->artifact_smoothing >= 0) || !(p->sharpen >= 0) || !isfinite(p->convergence))
        return fail(VSC_E_INVALID, "stereo parameter out of range");
    memset(g, 0, sizeof *g);
    g->height = H; g->width = W;
    const double total_buffer = 2.0 * p->max_disparity + fabs(p->convergence);
    const double stretch_factor = 1.0 + (total_buffer / (double)W);
    g->stretched_w = (int)((double)W * stretch_factor);
    g->super_sampled = p->super_sampling > 1.0;
    if (g->super_sampled) {
        g->ss_h = (int)((double)H * p->super_sampling);
        g->ss_w = (int)((double)g->stretched_w * p->super_sampling);
    } else {
        g->ss_h = H; g->ss_w = g->stretched_w;
    }
    const int base = (g->stretched_w - W) / 2;                    // both >= 0: floor division
    const int cs = (int)nearbyint(p->convergence);                 // Python round(): half to even
    const int lo = base + cs, ro = base - cs;
    if (g->super_sampled) {
        const double ratio = (double)g->ss_w / (double)g->stretched_w;
        g->left_crop = (int)((double)lo * ratio);
        g->right_crop = (int)((double)ro * ratio);
        g->crop_w = (int)((double)W * ratio);
    } else {
        g->left_crop = lo; g->right_crop = ro; g->crop_w = W;
    }
    if (p->edge_softness > 0) {
        int k = ((int)(p->edge_softness * 6)) | 1;
        k = k < 31 ? k : 31;
        g->blur_k = k > 5 ? k : 5;
    }
    if (p->artifact_smoothing > 0) {
        int d = (int)(p->artifact_smoothing * 4);
        d = d < 15 ? d : 15;
        g->bilateral_d = d > 5 ? d : 5;
    }
    if (lo < 0 || ro < 0)
        return fail(VSC_E_PARAMS, "convergence %.3f shifts a crop window left of the stretched view "
                    "(offsets %d/%d): the reference raises from _sharpen_image's reflect pad", p->convergence, lo, ro);
    if (g->crop_w < 3 || g->ss_h < 3)
        return fail(VSC_E_PARAMS, "cropped view too small for the 5x5 reflect pad");
    if (g->blur_k / 2 >= g->ss_h || g->blur_k / 2 >= g->ss_w)
        return fail(VSC_E_PARAMS, "depth blur kernel %d does not fit the %dx%d grid (reflect pad)", g->blur_k, g->ss_w, g->ss_h);
    if ((long long)g->ss_h * g->ss_w >= (1ll << 31))
        return fail(VSC_E_INVALID, "super-sampled grid exceeds 2^31 pixels");
    return VSC_OK;
}

// ------------------------------------------------------------------------------------------------
// context / slots
// ------------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return VSC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(VSC_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
        cap = want;
        return VSC_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Slot {
    cudaStream_t stream = nullptr;       // shared by the slots of one group (the group leader owns it)
    bool owns_stream = false;
    int nfr = 0;                         // leader only: frames in the group's current submission
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // inputs / outputs staged on device for host-buffer submissions
    DevBuf in_rgb, in_depth, out_sbs;
    // intermediates
    DevBuf rgb_st, depth_st, depth_ss, viewA[2], viewB[2], vmask[2];
    DevBuf st[2], tt[2], pstate[2], tile_u8[2], tile_i32[2], qkey[2], qidx[2];
    DevBuf tabs;        // lanczos + axis tables
    DevBuf scalars;     // FrameScalars
    DevBuf tstats;      // Telea phase counters (VSC_TELEA_STATS builds)
    DevBuf dp_scalars;  // min / max of the depth post-processing stage
    DevBuf png_work;    // PNG: filtered stream, segment blocks, segment metadata, file size
    DevBuf png_stage;   // PNG file of a submission whose host destination is pageable
    DevBuf png_stats;   // PNG debug counters (vsc_stage_png)
    FrameScalars* h_scalars = nullptr;   // pinned mirror
    unsigned long long* h_png = nullptr; // pinned: bytes of the PNG file of the last submission
    // table cache key
    int kH = 0, kW = 0, kSW = 0, kHs = 0, kWs = 0;
    const int* d_sx0 = nullptr; const short* d_it = nullptr; const float* d_ft = nullptr;
    const AxisTap* d_ty = nullptr; const AxisTap* d_tx = nullptr;
    int ib3 = 2048; float beta3 = 1.f;
    size_t qcap = 0;    // Telea queue capacity (entries per view)
    // last submission (for the overflow retry and for vsc_wait)
    bool busy = false;
    const uint8_t* l_rgb = nullptr; const void* l_depth = nullptr; uint8_t* l_out = nullptr;
    int l_dtype = 0, l_H = 0, l_W = 0; vsc_params l_p; uint8_t* l_host_out = nullptr; size_t l_out_bytes = 0;
    int l_layout = VSC_LAYOUT_SBS;       // output layout of the frame in this slot (fixed at submission)
    int l_pixfmt = VSC_PIXFMT_RGB24, l_matrix = VSC_MATRIX_BT709;   // its pixel format and YUV matrix (the same)
    int l_encode = VSC_ENCODE_NONE;      // its encoding (the same); with PNG, l_out holds the rgb24 frame and l_png the file
    uint8_t* l_png = nullptr;            // device-accessible destination of the PNG file
    const uint8_t* l_copy_src = nullptr; // device source of the copy into l_host_out (l_out_bytes bytes)
    int launches = 0;
    float last_ms = 0.f;
    bool done = false;                   // leader only: the stream has run past the submission (set by a host callback)
    struct vsc_ctx* owner = nullptr;
    bool prof = false;                   // per-kernel event pairs (vsc_set_profiling)
    // optional per-kernel profiling (vsc_set_profiling): event pairs around every launch
    std::vector<cudaEvent_t> pev;
    std::vector<const char*> pname;
    int pcount = 0;
};

struct vsc_ctx {
    int device = 0;
    int group_size = 1;                  // frames that share one stream and one hole-filling launch
    bool profiling = false;
    int layout = VSC_LAYOUT_SBS;         // output layout of frames submitted from now on (vsc_set_layout)
    int pixfmt = VSC_PIXFMT_RGB24;       // pixel format and YUV matrix of frames submitted from now on (vsc_set_pixfmt)
    int matrix = VSC_MATRIX_BT709;
    int encode = VSC_ENCODE_NONE;        // encoding of frames submitted from now on (vsc_set_encode)
    cudaStream_t tstream = nullptr;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    std::vector<cudaEvent_t> tslot;
    int sm_count = 148;
    std::vector<Slot> slots;
    std::mutex mu;                       // guards Slot::done; vsc_wait_any sleeps on cv until a submission completes
    std::condition_variable cv;
    DevBuf color_w;     // bilateral colour LUT for sigmaColor = 30 (stereo_core.py:410)
    DevBuf pow_tab;     // tables of the deterministic pow (apply_depth_gamma)
};

// The pow tables of the specification (DESIGN.md, float order; the CPU oracle has its own copy), computed with the same
// fixed series in IEEE double (this file is compiled with -ffp-contract=off; fma() is the correctly rounded one).
static double tab_log2(double x) {
    int e;
    double m = frexp(x, &e);
    if (m < 0.70710678118654752440) { m *= 2.0; e -= 1; }
    const double s = (m - 1.0) / (m + 1.0), z = s * s;
    double p = 1.0 / 27.0;
    for (int d = 25; d >= 1; d -= 2) p = fma(p, z, 1.0 / (double)d);
    const double ln_m = 2.0 * s * p;
    return fma(ln_m, 1.4426950408889634074, (double)e);
}
static double tab_exp2(double t) {
    const double n = nearbyint(t), f = (t - n) * 0.69314718055994530942;
    static const double inv_fact[14] = {1.0, 1.0, 1.0 / 2.0, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0, 1.0 / 720.0, 1.0 / 5040.0,
                                        1.0 / 40320.0, 1.0 / 362880.0, 1.0 / 3628800.0, 1.0 / 39916800.0,
                                        1.0 / 479001600.0, 1.0 / 6227020800.0};
    double p = inv_fact[13];
    for (int d = 12; d >= 0; d--) p = fma(p, f, inv_fact[d]);
    return ldexp(p, (int)n);
}
static void pow_tables(double* tab) {
    for (int i = 0; i < 128; i++) {
        const double c = 1.0 + ((double)i + 0.5) / 128.0;
        tab[i] = 1.0 / c;
        tab[128 + i] = tab_log2(c);
    }
    for (int j = 0; j < 64; j++) tab[256 + j] = tab_exp2((double)j / 64.0);
}

static int upload_constants(vsc_ctx* ctx) {
    TapConst tc;
    memset(&tc, 0, sizeof tc);
    int n = 0;
    for (int dk = -3; dk <= 3; dk++)
        for (int dl = -3; dl <= 3; dl++) {
            if (dk * dk + dl * dl > 9 || (dk == 0 && dl == 0)) continue;
            tc.dk[n] = (signed char)dk; tc.dl[n] = (signed char)dl;
            const float ry = (float)(-dk), rx = (float)(-dl);
            const float vl = rx * rx + ry * ry;
            tc.dst[n] = (float)(1. / ((double)vl * sqrt((double)vl)));
            n++;
        }
    CU(cudaMemcpyToSymbol(c_taps, &tc, sizeof tc));
    float cw[768];
    BilateralTaps bt;
    bilateral_tables(5, 30.0, 25.0, cw, bt);
    if (ctx->color_w.ensure(sizeof cw)) return VSC_E_NOMEM;
    CU(cudaMemcpy(ctx->color_w.p, cw, sizeof cw, cudaMemcpyHostToDevice));
    double pt[kPowTabN];
    pow_tables(pt);
    if (ctx->pow_tab.ensure(sizeof pt)) return VSC_E_NOMEM;
    CU(cudaMemcpy(ctx->pow_tab.p, pt, sizeof pt, cudaMemcpyHostToDevice));
    return VSC_OK;
}

template <int K, int P>
static int backend_attrs(int smem) {
    const void* f[] = {(const void*)backend_kernel<K, VSC_LAYOUT_SBS, P>, (const void*)backend_kernel<K, VSC_LAYOUT_HALF_SBS, P>,
                       (const void*)backend_kernel<K, VSC_LAYOUT_TB, P>, (const void*)backend_kernel<K, VSC_LAYOUT_HALF_TB, P>,
                       (const void*)backend_kernel<K, VSC_LAYOUT_ANAGLYPH, P>};
    for (const void* k : f) CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    return VSC_OK;
}
template <int K>
static int backend_attrs(int smem) {
    int rc;
    if ((rc = backend_attrs<K, VSC_PIXFMT_RGB24>(smem)) || (rc = backend_attrs<K, VSC_PIXFMT_YUV420P>(smem)) ||
        (rc = backend_attrs<K, VSC_PIXFMT_YUV420P10LE>(smem))) return rc;
    return VSC_OK;
}
static int set_smem_attrs() {
    const int big = 200 * 1024;
    CU(cudaFuncSetAttribute(lanczos_rgb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(lanczos_depth_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(lanczos_depth_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(lanczos_depth_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(depth_front_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(depth_front_kernel<31>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(warp_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(warp_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU(cudaFuncSetAttribute(warp_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    int rc;
    if ((rc = backend_attrs<0>(big)) || (rc = backend_attrs<2>(big)) || (rc = backend_attrs<3>(big)) || (rc = backend_attrs<4>(big))) return rc;
    CU(cudaFuncSetAttribute(telea_march_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MarchSh<16>)));
    CU(cudaFuncSetAttribute(telea_march_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MarchSh<32>)));
    CU(cudaFuncSetAttribute(png_segment_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PNG_SEG_SMEM));
    return VSC_OK;
}

extern "C" int vsc_create_grouped(int device, int n_groups, int group_size, vsc_ctx** out) {
    if (!out) return fail(VSC_E_INVALID, "null out pointer");
    *out = nullptr;
    if (n_groups < 1 || n_groups > 64) return fail(VSC_E_INVALID, "number of slots must be in [1,64]");
    if (group_size < 1 || group_size > TELEA_MAX_VIEWS / 2) return fail(VSC_E_INVALID, "group size must be in [1,%d]", TELEA_MAX_VIEWS / 2);
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);   // one hardware queue per slot stream (no effect once a context exists)
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(VSC_E_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(VSC_E_INVALID, "device %d out of range [0,%d)", device, ndev);
    CU(cudaSetDevice(device));
    vsc_ctx* ctx = new vsc_ctx();
    ctx->device = device;
    ctx->group_size = group_size;
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    int rc = set_smem_attrs();
    if (rc == VSC_OK) rc = upload_constants(ctx);
    if (rc != VSC_OK) { delete ctx; return rc; }
    ctx->slots.resize((size_t)n_groups * group_size);
    for (size_t i = 0; i < ctx->slots.size(); i++) {
        Slot& s = ctx->slots[i];
        s.owner = ctx;
        bool ok = true;
        if (i % group_size == 0) {
            ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess;
            s.owns_stream = ok;
        } else {
            s.stream = ctx->slots[i - i % group_size].stream;
        }
        ok = ok && cudaEventCreate(&s.ev0) == cudaSuccess && cudaEventCreate(&s.ev1) == cudaSuccess &&
             cudaMallocHost((void**)&s.h_scalars, sizeof(FrameScalars)) == cudaSuccess &&
             cudaMallocHost((void**)&s.h_png, sizeof(unsigned long long)) == cudaSuccess;
        if (!ok) {
            vsc_destroy(ctx);
            return fail(VSC_E_CUDA, "failed to create stream/events for a slot");
        }
        memset(s.h_scalars, 0, sizeof(FrameScalars));
        *s.h_png = 0;
    }
    *out = ctx;
    return VSC_OK;
}
extern "C" int vsc_create(int device, int n_slots, vsc_ctx** out) { return vsc_create_grouped(device, n_slots, 1, out); }
extern "C" int vsc_group_size(const vsc_ctx* ctx) { return ctx ? ctx->group_size : 0; }

extern "C" void vsc_destroy(vsc_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& s : ctx->slots) {
        DevBuf* bufs[] = {&s.in_rgb, &s.in_depth, &s.out_sbs, &s.rgb_st, &s.depth_st, &s.depth_ss, &s.viewA[0], &s.viewA[1],
                          &s.viewB[0], &s.viewB[1], &s.vmask[0], &s.vmask[1], &s.st[0], &s.st[1], &s.tt[0], &s.tt[1], &s.pstate[0], &s.pstate[1],
                          &s.tile_u8[0], &s.tile_u8[1], &s.tile_i32[0], &s.tile_i32[1], &s.qkey[0], &s.qkey[1],
                          &s.qidx[0], &s.qidx[1], &s.tabs, &s.scalars};
        for (DevBuf* b : bufs) b->release();
        s.tstats.release();
        s.dp_scalars.release();
        s.png_work.release();
        s.png_stage.release();
        s.png_stats.release();
        for (cudaEvent_t e : s.pev) cudaEventDestroy(e);
        if (s.h_scalars) cudaFreeHost(s.h_scalars);
        if (s.h_png) cudaFreeHost(s.h_png);
        if (s.ev0) cudaEventDestroy(s.ev0);
        if (s.ev1) cudaEventDestroy(s.ev1);
        if (s.stream && s.owns_stream) cudaStreamDestroy(s.stream);
    }
    for (cudaEvent_t e : ctx->tslot) cudaEventDestroy(e);
    if (ctx->t0) cudaEventDestroy(ctx->t0);
    if (ctx->t1) cudaEventDestroy(ctx->t1);
    if (ctx->tstream) cudaStreamDestroy(ctx->tstream);
    ctx->color_w.release();
    ctx->pow_tab.release();
    delete ctx;
}
extern "C" int vsc_device(const vsc_ctx* ctx) { return ctx ? ctx->device : -1; }
extern "C" int vsc_num_slots(const vsc_ctx* ctx) { return ctx ? (int)(ctx->slots.size() / ctx->group_size) : 0; }
extern "C" int vsc_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(VSC_E_INVALID, "null out pointer");
    CU(cudaMallocHost(out, bytes));
    return VSC_OK;
}
extern "C" int vsc_host_free(void* p) { if (p) CU(cudaFreeHost(p)); return VSC_OK; }

static size_t depth_elem(int dtype) { return dtype == VSC_DEPTH_U8 ? 1 : (dtype == VSC_DEPTH_U16 ? 2 : 4); }
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// upload the tap tables for a geometry into the slot (cached by geometry)
static int ensure_tables(Slot& s, const vsc_geom& g) {
    if (s.kH == g.height && s.kW == g.width && s.kSW == g.stretched_w && s.kHs == g.ss_h && s.kWs == g.ss_w && s.tabs.p)
        return VSC_OK;
    std::vector<int> sx0; std::vector<float> ft; std::vector<short> it;
    lanczos_tables(g.width, g.stretched_w, sx0, ft, it);
    std::vector<AxisTap> ty, tx;
    axis_table(g.height, g.ss_h, ty);
    axis_table(g.stretched_w, g.ss_w, tx);
    float beta[8];
    lanczos4_coeffs(0.f, beta);
    s.beta3 = beta[3];
    s.ib3 = sat_short(beta[3] * 2048.f);
    size_t o_sx0 = 0, o_ft = align_up(o_sx0 + sx0.size() * 4, 256), o_it = align_up(o_ft + ft.size() * 4, 256),
           o_ty = align_up(o_it + it.size() * 2, 256), o_tx = align_up(o_ty + ty.size() * sizeof(AxisTap), 256),
           total = o_tx + tx.size() * sizeof(AxisTap);
    // the slot's previous frame (if any) has completed: submit() waits for the slot before reuse
    int rc = s.tabs.ensure(total);
    if (rc) return rc;
    std::vector<uint8_t> blob(total, 0);
    memcpy(&blob[o_sx0], sx0.data(), sx0.size() * 4);
    memcpy(&blob[o_ft], ft.data(), ft.size() * 4);
    memcpy(&blob[o_it], it.data(), it.size() * 2);
    memcpy(&blob[o_ty], ty.data(), ty.size() * sizeof(AxisTap));
    memcpy(&blob[o_tx], tx.data(), tx.size() * sizeof(AxisTap));
    CU(cudaMemcpyAsync(s.tabs.p, blob.data(), total, cudaMemcpyHostToDevice, s.stream));
    CU(cudaStreamSynchronize(s.stream));   // blob is a temporary
    uint8_t* b = s.tabs.as<uint8_t>();
    s.d_sx0 = (const int*)(b + o_sx0); s.d_ft = (const float*)(b + o_ft); s.d_it = (const short*)(b + o_it);
    s.d_ty = (const AxisTap*)(b + o_ty); s.d_tx = (const AxisTap*)(b + o_tx);
    s.kH = g.height; s.kW = g.width; s.kSW = g.stretched_w; s.kHs = g.ss_h; s.kWs = g.ss_w;
    return VSC_OK;
}

static void prof_begin(Slot& s, const char* name) {
    if (!s.prof) return;
    while ((int)s.pev.size() < 2 * (s.pcount + 1)) { cudaEvent_t e; cudaEventCreate(&e); s.pev.push_back(e); }
    if ((int)s.pname.size() <= s.pcount) s.pname.resize(s.pcount + 1);
    s.pname[s.pcount] = name;
    cudaEventRecord(s.pev[2 * s.pcount], s.stream);
}
static void prof_end(Slot& s) {
    if (!s.prof) return;
    cudaEventRecord(s.pev[2 * s.pcount + 1], s.stream);
    s.pcount++;
}
#define KCHECK(s) do { cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) return fail(VSC_E_CUDA, "kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(e_)); (s).launches++; prof_end(s); } while (0)

// ---- device-level stage launchers (all asynchronous on s.stream) --------------------------------
static int run_lanczos_rgb(Slot& s, const uint8_t* d_rgb, int H, int W, int SW, uint8_t* d_out, FrameScalars* reset_fs = nullptr) {
    const int stage = (int)align_up((size_t)W * 3 + 32, 16);
    const size_t smem = stage + align_up((size_t)SW * 3 + 16, 16);
    if (smem > 200 * 1024) return fail(VSC_E_INVALID, "frame width %d too large for the row-staged Lanczos kernel", W);
    prof_begin(s, "lanczos_rgb_kernel");
    lanczos_rgb_kernel<<<H, kThreads, smem, s.stream>>>(d_rgb, W, SW, s.d_sx0, s.d_it, s.ib3, d_out, stage, reset_fs);
    KCHECK(s);
    return VSC_OK;
}
static int run_lanczos_depth(Slot& s, const void* d_depth, int dtype, int H, int W, int SW, float* d_out) {
    const size_t smem = align_up((size_t)W * depth_elem(dtype) + 32, 16);
    if (smem > 200 * 1024) return fail(VSC_E_INVALID, "frame width %d too large for the row-staged Lanczos kernel", W);
    FrameScalars* fs = s.scalars.as<FrameScalars>();
    prof_begin(s, "lanczos_depth_kernel");
    if (dtype == VSC_DEPTH_U8)
        lanczos_depth_kernel<uint8_t><<<H, kThreads, smem, s.stream>>>((const uint8_t*)d_depth, W, SW, s.d_sx0, s.d_it, s.d_ft, s.ib3, s.beta3, d_out, fs);
    else if (dtype == VSC_DEPTH_U16)
        lanczos_depth_kernel<uint16_t><<<H, kThreads, smem, s.stream>>>((const uint16_t*)d_depth, W, SW, s.d_sx0, s.d_it, s.d_ft, s.ib3, s.beta3, d_out, fs);
    else
        lanczos_depth_kernel<float><<<H, kThreads, smem, s.stream>>>((const float*)d_depth, W, SW, s.d_sx0, s.d_it, s.d_ft, s.ib3, s.beta3, d_out, fs);
    KCHECK(s);
    return VSC_OK;
}
static int run_depth_front(vsc_ctx* ctx, Slot& s, const vsc_geom& g, const vsc_params& p, float* d_depth_st, float* d_depth_ss) {
    const size_t n = (size_t)g.height * g.stretched_w;
    prof_begin(s, "normalize_kernel");
    normalize_kernel<<<ctx->sm_count * 4, kThreads, 0, s.stream>>>(d_depth_st, n, s.scalars.as<FrameScalars>());
    KCHECK(s);
    const int apply_gamma = p.depth_gamma != 1.0;
    const float gamma = (float)p.depth_gamma;
    if (g.blur_k > 0) {
        GaussTaps gt = gauss_taps(g.blur_k, p.edge_softness);
        const int r = g.blur_k / 2, AH = DF_T + 2 * r;
        // upsampled tile + horizontally blurred tile (also the staging area of the separable upsample) + row taps + pow tables
        const size_t smem = ((size_t)AH * AH + (size_t)AH * DF_SB) * 4 + (size_t)AH * sizeof(AxisTap) + kPowTabN * sizeof(double);
        dim3 grid((g.ss_w + DF_T - 1) / DF_T, (g.ss_h + DF_T - 1) / DF_T);
        prof_begin(s, "depth_front_kernel");
        if (g.blur_k == 31)
            depth_front_kernel<31><<<grid, kThreads, smem, s.stream>>>(d_depth_st, g.stretched_w, g.ss_h, g.ss_w, s.d_ty, s.d_tx,
                                                                       g.super_sampled, gt, gamma, apply_gamma, ctx->pow_tab.as<double>(), d_depth_ss);
        else
            depth_front_kernel<0><<<grid, kThreads, smem, s.stream>>>(d_depth_st, g.stretched_w, g.ss_h, g.ss_w, s.d_ty, s.d_tx,
                                                                      g.super_sampled, gt, gamma, apply_gamma, ctx->pow_tab.as<double>(), d_depth_ss);
    } else {
        dim3 grid((g.ss_w + kThreads * 4 - 1) / (kThreads * 4), g.ss_h);
        prof_begin(s, "depth_point_kernel");
        depth_point_kernel<<<grid, kThreads, 0, s.stream>>>(d_depth_st, g.stretched_w, g.ss_h, g.ss_w, s.d_ty, s.d_tx,
                                                            g.super_sampled, gamma, apply_gamma, ctx->pow_tab.as<double>(), d_depth_ss);
    }
    KCHECK(s);
    return VSC_OK;
}
static int run_warp(Slot& s, const vsc_geom& g, double max_disparity, const uint8_t* d_rgb_st, const float* d_depth_ss,
                    uchar4* vl, uchar4* vr, uint8_t* ml, uint8_t* mr, unsigned* hl, unsigned* hr, int mode) {
    WarpArgs a;
    a.rgb_st = d_rgb_st; a.depth = d_depth_ss; a.ty = s.d_ty; a.tx = s.d_tx;
    a.view[0] = vl; a.view[1] = vr; a.mask[0] = ml; a.mask[1] = mr;
    a.holes[0] = hl; a.holes[1] = hr; a.wb = (g.ss_w + 31) / 32;
    a.fs = s.scalars.as<FrameScalars>();
    a.H = g.height; a.SW = g.stretched_w; a.Hs = g.ss_h; a.Ws = g.ss_w;
    a.upsample = g.super_sampled;
    a.md = (float)max_disparity;
    a.R = (int)ceil(max_disparity) + 1;
    const int nseg = (g.ss_w + 1023) / 1024;
    a.TS = (int)align_up((size_t)(g.ss_w + nseg - 1) / nseg, 32);
    a.nseg = nseg;
    a.mode = mode;
    const int nsrc = a.TS + 2 * a.R + 8;
    const double ratio = a.upsample ? (double)g.stretched_w / (double)g.ss_w : 1.0;
    a.rgb_stage_bytes = (int)align_up((size_t)((int)(nsrc * ratio) + 8) * 3 + 32, 16);
    const size_t smem = 2 * ((size_t)a.TS + 1) * 8 + 128 + 2 * ((size_t)a.TS * 4 + 16) + 2 * (size_t)a.rgb_stage_bytes;
    dim3 grid(nseg, g.ss_h);
    prof_begin(s, "warp_kernel");
    switch (mode) {
        case 0: warp_kernel<0><<<grid, kThreads, smem, s.stream>>>(a); break;
        case 1: warp_kernel<1><<<dim3(std::min(nseg * g.ss_h, 592)), kThreads, smem, s.stream>>>(a); break;   // normally exits at once
        default: warp_kernel<2><<<grid, kThreads, smem, s.stream>>>(a); break;
    }
    KCHECK(s);
    return VSC_OK;
}
static int run_bilateral(vsc_ctx* ctx, Slot& s, int Hs, int Ws, double smoothing, const uchar4* in0, const uchar4* in1,
                         uchar4* out0, uchar4* out1, int nviews) {
    BilateralArgs a;
    int d = (int)(smoothing * 4);
    d = d < 15 ? d : 15;
    d = d > 5 ? d : 5;
    bilateral_tables(d, 30.0, smoothing * 25, nullptr, a.taps);
    a.in[0] = in0; a.in[1] = in1; a.out[0] = out0; a.out[1] = out1;
    a.color_w = ctx->color_w.as<float>();
    a.Hs = Hs; a.Ws = Ws;
    const int TW = 32 + 2 * a.taps.radius;
    const size_t smem = ((a.taps.radius == 2 ? 3 * 768 : 768) + (size_t)TW * TW) * 4;
    dim3 grid((Ws + 31) / 32, (Hs + 31) / 32, nviews), block(32, 8);
    prof_begin(s, "bilateral_kernel");
    switch (a.taps.radius) {
        case 2: bilateral_kernel<2><<<grid, block, smem, s.stream>>>(a); break;
        case 3: bilateral_kernel<3><<<grid, block, smem, s.stream>>>(a); break;
        case 4: bilateral_kernel<4><<<grid, block, smem, s.stream>>>(a); break;
        case 5: bilateral_kernel<5><<<grid, block, smem, s.stream>>>(a); break;
        case 6: bilateral_kernel<6><<<grid, block, smem, s.stream>>>(a); break;
        case 7: bilateral_kernel<7><<<grid, block, smem, s.stream>>>(a); break;
        default: return fail(VSC_E_INVALID, "bilateral radius %d not supported", a.taps.radius);
    }
    KCHECK(s);
    return VSC_OK;
}
// scratch of one eye of a frame slot; T / order words are skipped when the caller lends dead buffers for them
static int ensure_telea_view(Slot& s, int v, int Hs, int Ws, bool need_tt, bool need_pstate) {
    const size_t npx = (size_t)Hs * Ws;
    const int tw = (Ws + TG - 1) / TG, th = (Hs + TG - 1) / TG;
    const size_t nt = (size_t)tw * th;
    if (s.qcap == 0) s.qcap = npx / 8 > (1u << 20) ? npx / 8 : (1u << 20);
    if (s.qcap > npx + 1024) s.qcap = npx + 1024;
    int rc = 0;
    rc |= s.st[v].ensure(npx);
    if (need_tt) rc |= s.tt[v].ensure(npx * 4);
    if (need_pstate) rc |= s.pstate[v].ensure(npx * 4);
    rc |= s.tile_u8[v].ensure(nt * 2);
    rc |= s.tile_i32[v].ensure(nt * 4 * 11);
    rc |= s.qkey[v].ensure(s.qcap * 8 * 3);
    rc |= s.qidx[v].ensure(s.qcap * 4 * 3);
    return rc ? VSC_E_NOMEM : VSC_OK;
}
struct ViewSpec {       // one eye of one frame for the hole-filling launch
    Slot* fr;           // the frame slot that owns the scratch buffers and the frame scalars
    int b;              // 0 = left, 1 = right
    uchar4* img;
    const unsigned* holes;   // hole bitmap written by the warp kernel (or pack_holes_kernel)
    int k0, k1;         // columns the back end reads
    // Optional [Hs*Ws] 32-bit buffers lent for the arrival times T and the order words: buffers of the frame that are
    // dead by the time the hole filling starts (null = the slot's own scratch).  Only written / read near holes.
    float* tt = nullptr;
    unsigned* pstate = nullptr;
};
// `s` is the group leader (stream, launch / profiling bookkeeping); the views may belong to several frame slots
static int run_telea(vsc_ctx* ctx, Slot& s, int Hs, int Ws, const ViewSpec* vs, int nviews) {
    if (nviews < 1 || nviews > TELEA_MAX_VIEWS) return fail(VSC_E_INVALID, "bad view count");
    for (int v = 0; v < nviews; v++) { int rc = ensure_telea_view(*vs[v].fr, vs[v].b, Hs, Ws, !vs[v].tt, !vs[v].pstate); if (rc) return rc; }
    TeleaArgs a;
    memset(&a, 0, sizeof a);
    a.Hs = Hs; a.Ws = Ws; a.tw = (Ws + TG - 1) / TG; a.th = (Hs + TG - 1) / TG;
    a.nviews = nviews;
    a.wb = (Ws + 31) / 32;
#ifdef VSC_TELEA_STATS
    if (s.tstats.ensure(64 * 8)) return VSC_E_NOMEM;
    CU(cudaMemsetAsync(s.tstats.p, 0, 64 * 8, s.stream));
    a.stats = s.tstats.as<unsigned long long>();
#endif
    const size_t nt = (size_t)a.tw * a.th;
    for (int v = 0; v < nviews; v++) {
        Slot& f = *vs[v].fr;
        const int b = vs[v].b;
        TeleaView& V = a.v[v];
        V.img = vs[v].img; V.holes = vs[v].holes;
        V.st = f.st[b].as<uint8_t>(); V.tt = vs[v].tt ? vs[v].tt : f.tt[b].as<float>();
        V.tile_cnt = f.tile_u8[b].as<unsigned char>(); V.tile_need = V.tile_cnt + nt;
        int* ib = f.tile_i32[b].as<int>();
        V.lab = ib; V.csize = ib + nt; V.ctiles = ib + 2 * nt; V.cneed = ib + 3 * nt; V.cslot = ib + 4 * nt;
        V.cl_qoff = ib + 5 * nt; V.cl_toff = ib + 6 * nt; V.cl_ntiles = ib + 7 * nt; V.cl_size = ib + 8 * nt;
        V.cl_fill = ib + 9 * nt; V.tile_list = ib + 10 * nt;
        V.qkey[0] = f.qkey[b].as<unsigned long long>(); V.qkey[1] = V.qkey[0] + f.qcap; V.qkey[2] = V.qkey[1] + f.qcap;
        V.qidx[0] = f.qidx[b].as<unsigned>(); V.qidx[1] = V.qidx[0] + f.qcap; V.qidx[2] = V.qidx[1] + f.qcap;
        V.pstate = vs[v].pstate ? vs[v].pstate : f.pstate[b].as<unsigned>();
        V.qcap = (int)f.qcap;
        V.fs = f.scalars.as<FrameScalars>();
        V.vi = b;
        V.keep_x0 = vs[v].k0; V.keep_x1 = vs[v].k1;
    }
    // the prepare kernel also resets the dataflow words (pstate) within reach of a hole; the rest is never read
    dim3 pgrid((Ws + 31) / 32, (Hs + PR_ROWS * 8 - 1) / (PR_ROWS * 8), nviews), pblock(32, 8);
    prof_begin(s, "telea_prepare_kernel");
    telea_prepare_kernel<<<pgrid, pblock, 0, s.stream>>>(a);
    KCHECK(s);
    const int tb = (int)((nt + kThreads - 1) / kThreads);
    const int tgrid = tb < ctx->sm_count * 8 ? tb : ctx->sm_count * 8;
    prof_begin(s, "telea_ccl_init_kernel");
    telea_ccl_init_kernel<<<tgrid, kThreads, 0, s.stream>>>(a);    KCHECK(s);
    prof_begin(s, "telea_ccl_merge_kernel");
    telea_ccl_merge_kernel<<<tgrid, kThreads, 0, s.stream>>>(a);   KCHECK(s);
    prof_begin(s, "telea_ccl_flatten_kernel");
    telea_ccl_flatten_kernel<<<tgrid, kThreads, 0, s.stream>>>(a); KCHECK(s);
    prof_begin(s, "telea_cluster_alloc_kernel");
    telea_cluster_alloc_kernel<<<tgrid, kThreads, 0, s.stream>>>(a); KCHECK(s);
    prof_begin(s, "telea_cluster_fill_kernel");
    telea_cluster_fill_kernel<<<tgrid, kThreads, 0, s.stream>>>(a);  KCHECK(s);
#ifndef VSC_EXPERIMENT_NO_MARCH
    // persistent CTAs pulling clusters from a per-view queue (big clusters first); view-major launch order, so the
    // first CTAs to start take each view's biggest cluster
    dim3 cgrid(nviews, ctx->sm_count / 2);
    prof_begin(s, "telea_march_kernel");
    if (ctx->slots.size() == (size_t)ctx->group_size)     // one slot: nothing overlaps the march, favour its latency
        telea_march_kernel<32><<<cgrid, 32 * 32, sizeof(MarchSh<32>), s.stream>>>(a);
    else
        telea_march_kernel<16><<<cgrid, 16 * 32, sizeof(MarchSh<16>), s.stream>>>(a);
    KCHECK(s);
#endif
    return VSC_OK;
}
template <int K, int L>
static void launch_backend(int pixfmt, dim3 grid, size_t smem, cudaStream_t st, const BackendArgs& a) {
    switch (pixfmt) {
        case VSC_PIXFMT_YUV420P: backend_kernel<K, L, VSC_PIXFMT_YUV420P><<<grid, kThreads, smem, st>>>(a); break;
        case VSC_PIXFMT_YUV420P10LE: backend_kernel<K, L, VSC_PIXFMT_YUV420P10LE><<<grid, kThreads, smem, st>>>(a); break;
        default: backend_kernel<K, L, VSC_PIXFMT_RGB24><<<grid, kThreads, smem, st>>>(a); break;
    }
}
template <int K>
static void launch_backend(int layout, int pixfmt, dim3 grid, size_t smem, cudaStream_t st, const BackendArgs& a) {
    switch (layout) {
        case VSC_LAYOUT_HALF_SBS: launch_backend<K, VSC_LAYOUT_HALF_SBS>(pixfmt, grid, smem, st, a); break;
        case VSC_LAYOUT_TB: launch_backend<K, VSC_LAYOUT_TB>(pixfmt, grid, smem, st, a); break;
        case VSC_LAYOUT_HALF_TB: launch_backend<K, VSC_LAYOUT_HALF_TB>(pixfmt, grid, smem, st, a); break;
        case VSC_LAYOUT_ANAGLYPH: grid.z = 1; launch_backend<K, VSC_LAYOUT_ANAGLYPH>(pixfmt, grid, smem, st, a); break;
        default: launch_backend<K, VSC_LAYOUT_SBS>(pixfmt, grid, smem, st, a); break;
    }
}
// the YUV matrices of include/vsc_b200.h: rows cy, cu, cv in Q20 (BT.709 from Kr = 0.2126, Kb = 0.0722; BT.601 is
// OpenCV's RGB2YUV_I420 table)
static const int kYuvMatrix[2][9] = {
    {191455, 644068, 65019, -105533, -355018, 460551, 460551, -418321, -42230},
    {269484, 528482, 102760, -155188, -305135, 460324, 460324, -385875, -74448},
};
// d_out holds the frame in `layout` and `pixfmt` (vsc_output_size; the caller has checked that they take H x W)
static int run_backend(Slot& s, const vsc_geom& g, double sharpen, const uchar4* v0, const uchar4* v1, uint8_t* d_out,
                       int layout, int pixfmt = VSC_PIXFMT_RGB24, int matrix = VSC_MATRIX_BT709) {
    BackendArgs a;
    memcpy(a.yuv, kYuvMatrix[matrix], sizeof a.yuv);
    a.view[0] = v0; a.view[1] = v1; a.out = d_out;
    a.H = g.height; a.W = g.width; a.Hs = g.ss_h; a.Ws = g.ss_w;
    a.crop[0] = g.left_crop; a.crop[1] = g.right_crop; a.cw = g.crop_w;
    // integer super-sampling (the usual case): compile-time tile geometry
    int K = 0;
    for (int k = 2; k <= 4; k++) if (g.ss_h == k * g.height && g.crop_w == k * g.width) K = k;
    a.RH = K ? BE_OY * K : (int)(((long long)BE_OY * g.ss_h + g.height - 1) / g.height) + 1;
    a.RW = K ? BE_OX * K + 1 : (int)(((long long)BE_OX * g.crop_w + g.width - 1) / g.width) + 1;
    a.strength = (float)sharpen;
    a.do_sharpen = sharpen > 0;
    a.g5 = gauss_taps(5, 1.0);
    // staged input + horizontally blurred planes (+ sharpened planes unless K == 3 pools from registers) + output bytes
    const size_t smem = (size_t)(a.RH + 4) * (a.RW + 4) * 4 + (size_t)3 * (a.RH + 4) * a.RW * 4 +
                        (K == 3 ? 0 : (size_t)3 * a.RH * a.RW * 4) + (size_t)BE_OY * (BE_OX * 3 + 16);
    if (smem > 200 * 1024) return fail(VSC_E_INVALID, "super_sampling too large for the back-end tile (%zu bytes of shared memory)", smem);
    dim3 grid((g.width + BE_OX - 1) / BE_OX, (g.height + BE_OY - 1) / BE_OY, 2);
    prof_begin(s, "backend_kernel");
    switch (K) {       // the anaglyph runs both eyes in one CTA (grid.z = 1)
        case 2: launch_backend<2>(layout, pixfmt, grid, smem, s.stream, a); break;
        case 3: launch_backend<3>(layout, pixfmt, grid, smem, s.stream, a); break;
        case 4: launch_backend<4>(layout, pixfmt, grid, smem, s.stream, a); break;
        default: launch_backend<0>(layout, pixfmt, grid, smem, s.stream, a); break;
    }
    KCHECK(s);
    return VSC_OK;
}

// PNG encoding (vsc_png.cuh): filtered stream, one deflate segment per PNG_SEG bytes of it, worst-case file bytes
static size_t png_stream_bytes(int oh, int ow) { return (size_t)oh * (1 + 3 * (size_t)ow); }
static size_t png_segments(int oh, int ow) { return (png_stream_bytes(oh, ow) + PNG_SEG - 1) / PNG_SEG; }
static size_t png_capacity(int oh, int ow) { return 53 + png_stream_bytes(oh, ow) + 22 * png_segments(oh, ow); }
// Encode the rgb24 frames (oh x ow) that fr[0..n) hold at l_out into PNG files at fr[i].l_png (device-accessible);
// three launches on the leader's stream for the whole group.  The file sizes land in fr[i].h_png once the stream
// has run.  stats: null, or the 3 debug counters of png_segment_kernel.
static int run_png(Slot& lead, Slot* fr, int n, int oh, int ow, unsigned long long* stats) {
    const size_t N = png_stream_bytes(oh, ow), nseg = png_segments(oh, ow);
    if (nseg > (size_t)(1 << 30)) return fail(VSC_E_INVALID, "frame %dx%d too large for PNG output", ow, oh);
    PngArgs a;
    memset(&a, 0, sizeof a);
    a.oh = oh; a.ow = ow; a.n = (long long)N; a.nseg = (int)nseg; a.stats = stats;
    const size_t o_seg = align_up(N, 256), o_meta = o_seg + nseg * PNG_SEG_STRIDE,
                 o_size = o_meta + align_up(nseg * sizeof(PngSegMeta), 256);
    for (int i = 0; i < n; i++) {
        if (fr[i].png_work.ensure(o_size + 256)) return VSC_E_NOMEM;
        uint8_t* b = fr[i].png_work.as<uint8_t>();
        a.img[i] = fr[i].l_out; a.dst[i] = fr[i].l_png;
        a.filt[i] = b; a.seg[i] = b + o_seg; a.meta[i] = (PngSegMeta*)(b + o_meta); a.size[i] = (unsigned long long*)(b + o_size);
    }
    prof_begin(lead, "png_filter_kernel");
    png_filter_kernel<<<dim3(oh, n), 256, 0, lead.stream>>>(a);
    KCHECK(lead);
    prof_begin(lead, "png_segment_kernel");
    png_segment_kernel<<<dim3((unsigned)nseg, n), PNG_SEG_THREADS, PNG_SEG_SMEM, lead.stream>>>(a);
    KCHECK(lead);
    prof_begin(lead, "png_assemble_kernel");
    png_assemble_kernel<<<dim3((unsigned)nseg, n), 256, 0, lead.stream>>>(a);
    KCHECK(lead);
    for (int i = 0; i < n; i++)
        CU(cudaMemcpyAsync(fr[i].h_png, a.size[i], sizeof(unsigned long long), cudaMemcpyDeviceToHost, lead.stream));
    return VSC_OK;
}

// ---- whole frame ----------------------------------------------------------------------------------
static int ensure_frame_buffers(Slot& s, const vsc_geom& g, bool smoothing) {
    const size_t npx = (size_t)g.ss_h * g.ss_w;
    int rc = 0;
    rc |= s.scalars.ensure(sizeof(FrameScalars));
    rc |= s.rgb_st.ensure((size_t)g.height * g.stretched_w * 3);
    rc |= s.depth_st.ensure((size_t)g.height * g.stretched_w * 4);
    rc |= s.depth_ss.ensure(npx * 4);
    for (int v = 0; v < 2; v++) {
        rc |= s.viewA[v].ensure(npx * 4);
        if (smoothing) rc |= s.viewB[v].ensure(npx * 4);
        rc |= s.vmask[v].ensure((size_t)g.ss_h * ((g.ss_w + 31) / 32) * 4);     // hole bitmap, 1 bit per pixel
    }
    return rc ? VSC_E_NOMEM : VSC_OK;
}

// Enqueue n frames of one group (slot) on the group's stream.  Every frame runs its own wide kernels; the
// hole filling of all frames is ONE launch sequence, so that the latency-bound march of up to
// group_size frames overlaps on a single stream.  `fr` points at the group's first frame slot (the leader).
static int enqueue_group(vsc_ctx* ctx, Slot* fr, int n, int dtype, const vsc_geom& g, const vsc_params& p) {
    Slot& lead = fr[0];
    const bool smoothing = p.artifact_smoothing > 0;
    for (int i = 0; i < n; i++) {
        int rc = ensure_frame_buffers(fr[i], g, smoothing);
        if (!rc) rc = ensure_tables(fr[i], g);
        if (rc) return rc;
        fr[i].launches = 0;
        fr[i].pcount = 0;
    }
    CU(cudaEventRecord(lead.ev0, lead.stream));
    ViewSpec vs[TELEA_MAX_VIEWS];
    uchar4* cur[TELEA_MAX_VIEWS];
    for (int i = 0; i < n; i++) {
        Slot& s = fr[i];
        int rc;
        if ((rc = run_lanczos_rgb(s, s.l_rgb, g.height, g.width, g.stretched_w, s.rgb_st.as<uint8_t>(), s.scalars.as<FrameScalars>()))) return rc;
        if ((rc = run_lanczos_depth(s, s.l_depth, dtype, g.height, g.width, g.stretched_w, s.depth_st.as<float>()))) return rc;
        if ((rc = run_depth_front(ctx, s, g, p, s.depth_st.as<float>(), s.depth_ss.as<float>()))) return rc;
        uchar4* va[2] = {s.viewA[0].as<uchar4>(), s.viewA[1].as<uchar4>()};
        unsigned* vm[2] = {s.vmask[0].as<unsigned>(), s.vmask[1].as<unsigned>()};     // hole bitmaps
        if ((rc = run_warp(s, g, p.max_disparity, s.rgb_st.as<uint8_t>(), s.depth_ss.as<float>(), va[0], va[1], nullptr, nullptr, vm[0], vm[1], 0))) return rc;
        cur[2 * i] = va[0]; cur[2 * i + 1] = va[1];
        if (smoothing) {
            // `if image_np.max() > 1.0 ... else (image_np * 255)` (stereo_core.py:404-407): conditional re-run on device
            if ((rc = run_warp(s, g, p.max_disparity, s.rgb_st.as<uint8_t>(), s.depth_ss.as<float>(), va[0], va[1], nullptr, nullptr, vm[0], vm[1], 1))) return rc;
            uchar4* vb[2] = {s.viewB[0].as<uchar4>(), s.viewB[1].as<uchar4>()};
            if ((rc = run_bilateral(ctx, s, g.ss_h, g.ss_w, p.artifact_smoothing, va[0], va[1], vb[0], vb[1], 2))) return rc;
            cur[2 * i] = vb[0]; cur[2 * i + 1] = vb[1];
        }
        vs[2 * i] = ViewSpec{&s, 0, cur[2 * i], vm[0], g.left_crop, g.left_crop + g.crop_w};
        vs[2 * i + 1] = ViewSpec{&s, 1, cur[2 * i + 1], vm[1], g.right_crop, g.right_crop + g.crop_w};
        if (smoothing) {
            // HBM capacity bounds the frames in flight (3.6 GB per 4K frame): the pre-bilateral views and the depth
            // map are dead once the bilateral filter has run, so they serve as T (both eyes) and order words (left eye)
            vs[2 * i].tt = s.viewA[0].as<float>();
            vs[2 * i + 1].tt = s.viewA[1].as<float>();
            vs[2 * i].pstate = s.depth_ss.as<unsigned>();
        }
    }
    int rc = run_telea(ctx, lead, g.ss_h, g.ss_w, vs, 2 * n);
    if (rc) return rc;
    for (int i = 0; i < n; i++)
        if ((rc = run_backend(fr[i], g, p.sharpen, cur[2 * i], cur[2 * i + 1], fr[i].l_out, fr[i].l_layout,
                                  fr[i].l_pixfmt, fr[i].l_matrix))) return rc;
    if (lead.l_encode == VSC_ENCODE_PNG) {
        int oh, ow;
        if ((rc = vsc_layout_shape(lead.l_layout, g.height, g.width, &oh, &ow)) || (rc = run_png(lead, fr, n, oh, ow, nullptr))) return rc;
    }
    CU(cudaEventRecord(lead.ev1, lead.stream));
    for (int i = 0; i < n; i++)
        CU(cudaMemcpyAsync(fr[i].h_scalars, fr[i].scalars.p, sizeof(FrameScalars), cudaMemcpyDeviceToHost, lead.stream));
    return VSC_OK;
}

static void CUDART_CB on_submission_done(void* p) {       // runs on a driver thread once the stream reaches it; no CUDA calls here
    Slot* lead = static_cast<Slot*>(p);
    {
        std::lock_guard<std::mutex> lk(lead->owner->mu);
        lead->done = true;
    }
    lead->owner->cv.notify_all();
}

// copies of the submission's outputs into caller-owned host buffers
static int enqueue_d2h(Slot* fr, int n) {
    for (int i = 0; i < n; i++)
        if (fr[i].l_host_out) CU(cudaMemcpyAsync(fr[i].l_host_out, fr[i].l_copy_src, fr[i].l_out_bytes, cudaMemcpyDeviceToHost, fr[0].stream));
    return VSC_OK;
}

static int submit_group_impl(vsc_ctx* ctx, int slot, int n, const uint8_t* const* rgb, const void* const* depth, int dtype,
                             int H, int W, const vsc_params* p, uint8_t* const* out, bool device_io) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    const int G = ctx->group_size;
    if (slot < 0 || slot >= (int)ctx->slots.size() / G) return fail(VSC_E_INVALID, "slot %d out of range", slot);
    if (n < 1 || n > G) return fail(VSC_E_INVALID, "a slot of this context takes 1..%d frames per submission", G);
    if (!rgb || !depth || !p || !out) return fail(VSC_E_INVALID, "null buffer");
    for (int i = 0; i < n; i++) if (!rgb[i] || !depth[i] || !out[i]) return fail(VSC_E_INVALID, "null buffer");
    if (dtype != VSC_DEPTH_U8 && dtype != VSC_DEPTH_U16 && dtype != VSC_DEPTH_F32) return fail(VSC_E_INVALID, "unsupported depth dtype %d", dtype);
    Slot* fr = &ctx->slots[(size_t)slot * G];
    Slot& lead = fr[0];
    if (lead.busy) return fail(VSC_E_STATE, "slot %d still has frames in flight; call vsc_wait first", slot);
    vsc_geom g;
    int rc;
    if ((rc = vsc_geometry(H, W, p, &g))) return rc;
    const int layout = ctx->layout, pixfmt = ctx->pixfmt, matrix = ctx->matrix, encode = ctx->encode;
    size_t nout, cap = 0;
    if ((rc = vsc_output_size(layout, pixfmt, H, W, &nout))) return rc;
    if (encode == VSC_ENCODE_PNG) {
        if (pixfmt != VSC_PIXFMT_RGB24) return fail(VSC_E_INVALID, "PNG output needs the rgb24 pixel format");
        if ((rc = vsc_encoded_capacity(layout, encode, H, W, &cap))) return rc;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t nrgb = (size_t)H * W * 3, ndepth = (size_t)H * W * depth_elem(dtype);
    for (int i = 0; i < n; i++) {
        Slot& s = fr[i];
        s.l_rgb = rgb[i]; s.l_depth = depth[i]; s.l_out = out[i]; s.l_host_out = nullptr; s.l_out_bytes = nout;
        s.l_layout = layout; s.l_pixfmt = pixfmt; s.l_matrix = matrix; s.l_encode = encode; s.l_png = nullptr;
        if (!device_io) {
            if (s.in_rgb.ensure(nrgb) || s.in_depth.ensure(ndepth) || s.out_sbs.ensure(nout)) return VSC_E_NOMEM;
            CU(cudaMemcpyAsync(s.in_rgb.p, rgb[i], nrgb, cudaMemcpyHostToDevice, lead.stream));
            CU(cudaMemcpyAsync(s.in_depth.p, depth[i], ndepth, cudaMemcpyHostToDevice, lead.stream));
            s.l_rgb = s.in_rgb.as<uint8_t>(); s.l_depth = s.in_depth.p; s.l_out = s.out_sbs.as<uint8_t>();
            s.l_host_out = out[i]; s.l_copy_src = s.l_out;
        }
        if (encode == VSC_ENCODE_PNG) {
            // the frame goes to the slot's own buffer, the file to the caller's: page-locked host memory is written by
            // the device directly (only the file's bytes cross the bus); a pageable one gets the capacity after the run
            if (device_io) {
                if (s.out_sbs.ensure(nout)) return VSC_E_NOMEM;
                s.l_png = out[i]; s.l_out = s.out_sbs.as<uint8_t>();
            } else {
                cudaPointerAttributes at;
                if (cudaPointerGetAttributes(&at, out[i]) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
                    s.l_png = (uint8_t*)at.devicePointer; s.l_host_out = nullptr;
                } else {
                    cudaGetLastError();
                    if (s.png_stage.ensure(cap)) return VSC_E_NOMEM;
                    s.l_png = s.png_stage.as<uint8_t>(); s.l_copy_src = s.l_png; s.l_out_bytes = cap;
                }
            }
        }
    }
    rc = enqueue_group(ctx, fr, n, dtype, g, *p);
    if (!rc) rc = enqueue_d2h(fr, n);
    if (rc) { cudaStreamSynchronize(lead.stream); return rc; }
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        lead.done = false;
    }
    CU(cudaLaunchHostFunc(lead.stream, on_submission_done, &lead));
    lead.busy = true;
    lead.nfr = n;
    lead.l_dtype = dtype; lead.l_H = H; lead.l_W = W; lead.l_p = *p;
    return VSC_OK;
}

extern "C" int vsc_submit_group(vsc_ctx* ctx, int slot, int n, const uint8_t* const* rgb, const void* const* depth, int dtype,
                                int H, int W, const vsc_params* p, uint8_t* const* out) {
    return submit_group_impl(ctx, slot, n, rgb, depth, dtype, H, W, p, out, false);
}
extern "C" int vsc_submit_device_group(vsc_ctx* ctx, int slot, int n, const uint8_t* const* d_rgb, const void* const* d_depth,
                                       int dtype, int H, int W, const vsc_params* p, uint8_t* const* d_out) {
    return submit_group_impl(ctx, slot, n, d_rgb, d_depth, dtype, H, W, p, d_out, true);
}
extern "C" int vsc_submit(vsc_ctx* ctx, int slot, const uint8_t* rgb, const void* depth, int dtype, int H, int W,
                          const vsc_params* p, uint8_t* out) {
    return submit_group_impl(ctx, slot, 1, &rgb, &depth, dtype, H, W, p, &out, false);
}
extern "C" int vsc_submit_device(vsc_ctx* ctx, int slot, const uint8_t* d_rgb, const void* d_depth, int dtype, int H, int W,
                                 const vsc_params* p, uint8_t* d_out) {
    return submit_group_impl(ctx, slot, 1, &d_rgb, &d_depth, dtype, H, W, p, &d_out, true);
}

static Slot* group_lead(vsc_ctx* ctx, int slot) {
    if (!ctx || slot < 0 || slot >= (int)ctx->slots.size() / ctx->group_size) return nullptr;
    return &ctx->slots[(size_t)slot * ctx->group_size];
}

extern "C" int vsc_wait(vsc_ctx* ctx, int slot) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr) return fail(VSC_E_INVALID, "bad context or slot");
    Slot& lead = fr[0];
    if (!lead.busy) return fail(VSC_E_STATE, "slot %d has no frame in flight", slot);
    CU(cudaSetDevice(ctx->device));
    const int n = lead.nfr;
    bool overflow = false;
    for (int attempt = 0; attempt < 4; attempt++) {
        cudaError_t e = cudaStreamSynchronize(lead.stream);
        if (e != cudaSuccess) { lead.busy = false; return fail(VSC_E_CUDA, "stream synchronize failed: %s", cudaGetErrorString(e)); }
        overflow = false;
        for (int i = 0; i < n; i++) {
            if (fr[i].h_scalars->overflow == 0x7fffffff) {      // raised by the march itself, never by a size
                lead.busy = false;
                return fail(VSC_E_STATE, "internal invariant of the hole-filling march violated (bucket range); please report the frame");
            }
            if (fr[i].h_scalars->overflow) {
                // Telea queue scratch was too small for this frame's holes: grow it and redo the submission
                const size_t need = (size_t)fr[i].h_scalars->overflow;
                fr[i].qcap = need + need / 4 + 1024;
                overflow = true;
            }
        }
        if (!overflow) break;
        vsc_geom g;
        int rc = vsc_geometry(lead.l_H, lead.l_W, &lead.l_p, &g);
        if (!rc) rc = enqueue_group(ctx, fr, n, lead.l_dtype, g, lead.l_p);
        if (!rc) rc = enqueue_d2h(fr, n);
        if (rc) { lead.busy = false; return rc; }
    }
    lead.busy = false;
    if (overflow) return fail(VSC_E_NOMEM, "hole-filling scratch overflow persisted");
    cudaEventElapsedTime(&lead.last_ms, lead.ev0, lead.ev1);
    return VSC_OK;
}

extern "C" int vsc_query(vsc_ctx* ctx, int slot) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr) return fail(VSC_E_INVALID, "bad context or slot");
    if (!fr->busy) return fail(VSC_E_STATE, "slot %d has no frame in flight", slot);
    cudaError_t e = cudaStreamQuery(fr->stream);
    if (e == cudaSuccess) return 1;
    if (e == cudaErrorNotReady) return 0;
    return fail(VSC_E_CUDA, "stream query failed: %s", cudaGetErrorString(e));
}

extern "C" int vsc_wait_any(vsc_ctx* ctx, const int* slots, int n, int timeout_ms, int* which) {
    if (!ctx || !slots || !which || n < 1) return fail(VSC_E_INVALID, "bad argument");
    *which = -1;
    for (int i = 0; i < n; i++) {
        Slot* fr = group_lead(ctx, slots[i]);
        if (!fr) return fail(VSC_E_INVALID, "slot %d out of range", slots[i]);
        if (!fr->busy) return fail(VSC_E_STATE, "slot %d has no frame in flight", slots[i]);
    }
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms < 0 ? 0 : timeout_ms);
    std::unique_lock<std::mutex> lk(ctx->mu);
    while (true) {
        for (int i = 0; i < n; i++)
            if (group_lead(ctx, slots[i])->done) { *which = slots[i]; return VSC_OK; }
        if (timeout_ms < 0) ctx->cv.wait(lk);
        else if (ctx->cv.wait_until(lk, deadline) == std::cv_status::timeout) return VSC_OK;      // *which stays -1
    }
}

extern "C" int vsc_sync(vsc_ctx* ctx) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    int rc = VSC_OK;
    for (int i = 0; i < (int)ctx->slots.size() / ctx->group_size; i++)
        if (group_lead(ctx, i)->busy) { int r = vsc_wait(ctx, i); if (r) rc = r; }
    return rc;
}
extern "C" void* vsc_slot_stream(vsc_ctx* ctx, int slot) {
    Slot* fr = group_lead(ctx, slot);
    return fr ? (void*)fr->stream : nullptr;
}
extern "C" int vsc_slot_elapsed_ms(vsc_ctx* ctx, int slot, float* ms) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr || !ms) return fail(VSC_E_INVALID, "bad argument");
    *ms = fr->last_ms;
    return VSC_OK;
}
extern "C" int vsc_slot_launches(vsc_ctx* ctx, int slot) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr) return -1;
    int total = 0;
    for (int i = 0; i < ctx->group_size; i++) total += fr[i].launches;
    return total;
}

extern "C" int vsc_layout_shape(int layout, int H, int W, int* out_h, int* out_w) {
    if (!out_h || !out_w) return fail(VSC_E_INVALID, "null argument");
    if (H < 1 || W < 1) return fail(VSC_E_INVALID, "bad frame size %dx%d", W, H);
    switch (layout) {
        case VSC_LAYOUT_SBS: *out_h = H; *out_w = 2 * W; return VSC_OK;
        case VSC_LAYOUT_TB: *out_h = 2 * H; *out_w = W; return VSC_OK;
        case VSC_LAYOUT_ANAGLYPH: *out_h = H; *out_w = W; return VSC_OK;
        case VSC_LAYOUT_HALF_SBS:
            if (W % 2) return fail(VSC_E_INVALID, "half-sbs halves the width: frame width %d is odd", W);
            *out_h = H; *out_w = W; return VSC_OK;
        case VSC_LAYOUT_HALF_TB:
            if (H % 2) return fail(VSC_E_INVALID, "half-tb halves the height: frame height %d is odd", H);
            *out_h = H; *out_w = W; return VSC_OK;
        default: return fail(VSC_E_INVALID, "unknown output layout %d", layout);
    }
}
extern "C" int vsc_set_layout(vsc_ctx* ctx, int layout) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    if (layout < VSC_LAYOUT_SBS || layout > VSC_LAYOUT_ANAGLYPH) return fail(VSC_E_INVALID, "unknown output layout %d", layout);
    ctx->layout = layout;
    return VSC_OK;
}
extern "C" int vsc_output_size(int layout, int pixfmt, int H, int W, size_t* bytes) {
    if (!bytes) return fail(VSC_E_INVALID, "null argument");
    int oh, ow, rc;
    if ((rc = vsc_layout_shape(layout, H, W, &oh, &ow))) return rc;
    const size_t n = (size_t)oh * ow;
    switch (pixfmt) {
        case VSC_PIXFMT_RGB24: *bytes = n * 3; return VSC_OK;
        case VSC_PIXFMT_YUV420P: case VSC_PIXFMT_YUV420P10LE: break;
        default: return fail(VSC_E_INVALID, "unknown pixel format %d", pixfmt);
    }
    // 4:2:0 needs whole 2x2 blocks, and each eye must start on an even coordinate of the output frame
    if (H % 2 || W % 2) return fail(VSC_E_INVALID, "yuv420 needs an even frame size: %dx%d", W, H);
    if (layout == VSC_LAYOUT_HALF_SBS && W % 4) return fail(VSC_E_INVALID, "yuv420 with half-sbs needs a width divisible by 4: %d", W);
    if (layout == VSC_LAYOUT_HALF_TB && H % 4) return fail(VSC_E_INVALID, "yuv420 with half-tb needs a height divisible by 4: %d", H);
    *bytes = pixfmt == VSC_PIXFMT_YUV420P ? n * 3 / 2 : n * 3;
    return VSC_OK;
}
extern "C" int vsc_set_pixfmt(vsc_ctx* ctx, int pixfmt, int matrix) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    if (pixfmt < VSC_PIXFMT_RGB24 || pixfmt > VSC_PIXFMT_YUV420P10LE) return fail(VSC_E_INVALID, "unknown pixel format %d", pixfmt);
    if (matrix < VSC_MATRIX_BT709 || matrix > VSC_MATRIX_BT601) return fail(VSC_E_INVALID, "unknown yuv matrix %d", matrix);
    if (ctx->encode == VSC_ENCODE_PNG && pixfmt != VSC_PIXFMT_RGB24)
        return fail(VSC_E_INVALID, "PNG output needs the rgb24 pixel format: set the encoding to none first");
    ctx->pixfmt = pixfmt;
    ctx->matrix = matrix;
    return VSC_OK;
}

extern "C" int vsc_encoded_capacity(int layout, int encode, int H, int W, size_t* bytes) {
    if (!bytes) return fail(VSC_E_INVALID, "null argument");
    if (encode == VSC_ENCODE_NONE) return vsc_output_size(layout, VSC_PIXFMT_RGB24, H, W, bytes);
    if (encode != VSC_ENCODE_PNG) return fail(VSC_E_INVALID, "unknown encoding %d", encode);
    int oh, ow, rc;
    if ((rc = vsc_layout_shape(layout, H, W, &oh, &ow))) return rc;
    *bytes = png_capacity(oh, ow);
    return VSC_OK;
}
extern "C" int vsc_set_encode(vsc_ctx* ctx, int encode) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    if (encode != VSC_ENCODE_NONE && encode != VSC_ENCODE_PNG) return fail(VSC_E_INVALID, "unknown encoding %d", encode);
    if (encode == VSC_ENCODE_PNG && ctx->pixfmt != VSC_PIXFMT_RGB24)
        return fail(VSC_E_INVALID, "PNG output needs the rgb24 pixel format");
    ctx->encode = encode;
    return VSC_OK;
}
extern "C" int vsc_encoded_bytes(vsc_ctx* ctx, int slot, int index, size_t* bytes) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr || !bytes) return fail(VSC_E_INVALID, "bad argument");
    if (fr->busy) return fail(VSC_E_STATE, "slot %d still has frames in flight; call vsc_wait first", slot);
    if (index < 0 || index >= fr->nfr) return fail(VSC_E_INVALID, "frame %d is not part of slot %d's last submission", index, slot);
    if (fr[index].l_encode != VSC_ENCODE_PNG) return fail(VSC_E_STATE, "slot %d's last submission was not encoded", slot);
    *bytes = (size_t)*fr[index].h_png;
    return VSC_OK;
}

extern "C" int vsc_process_frame(vsc_ctx* ctx, const uint8_t* rgb, const void* depth, int dtype, int H, int W,
                                 const vsc_params* p, uint8_t* out) {
    int rc = vsc_submit(ctx, 0, rgb, depth, dtype, H, W, p, out);
    if (rc) return rc;
    return vsc_wait(ctx, 0);
}

// ------------------------------------------------------------------------------------------------
// stage-level entry points (synchronous, host buffers) for per-stage parity tests
// ------------------------------------------------------------------------------------------------
struct Tmp {   // scoped device allocation
    void* p = nullptr;
    ~Tmp() { if (p) cudaFree(p); }
    int alloc(size_t n) { return cudaMalloc(&p, n ? n : 1) == cudaSuccess ? 0 : fail(VSC_E_NOMEM, "cudaMalloc(%zu) failed", n); }
};
#define STAGE_BEGIN()                                                   \
    if (!ctx) return fail(VSC_E_INVALID, "null context");               \
    Slot& s = ctx->slots[0];                                            \
    if (s.busy) return fail(VSC_E_STATE, "slot 0 busy");                \
    CU(cudaSetDevice(ctx->device));                                     \
    if (s.scalars.ensure(sizeof(FrameScalars))) return VSC_E_NOMEM;     \
    frame_init_kernel<<<1, 32, 0, s.stream>>>(s.scalars.as<FrameScalars>());

static vsc_geom stage_geom(int H, int W, int SW, int Hs, int Ws) {
    vsc_geom g;
    memset(&g, 0, sizeof g);
    g.height = H; g.width = W; g.stretched_w = SW; g.ss_h = Hs; g.ss_w = Ws;
    g.super_sampled = !(Hs == H && Ws == SW);
    return g;
}

extern "C" int vsc_stage_lanczos(vsc_ctx* ctx, const void* src, int dtype, int channels, int H, int W, int dW, void* dst) {
    STAGE_BEGIN();
    if (!src || !dst || H < 1 || W < 1 || dW < 1) return fail(VSC_E_INVALID, "bad argument");
    if (!((dtype == VSC_DEPTH_U8 && (channels == 1 || channels == 3)) || (channels == 1 && (dtype == VSC_DEPTH_U16 || dtype == VSC_DEPTH_F32))))
        return fail(VSC_E_INVALID, "unsupported dtype/channels");
    vsc_geom g = stage_geom(H, W, dW, H, dW);
    s.kH = 0;   // force table rebuild (W may differ from the cached key's semantics)
    int rc = ensure_tables(s, g);
    if (rc) return rc;
    const size_t es = depth_elem(dtype), nin = (size_t)H * W * channels * es;
    Tmp din, dout;
    if (din.alloc(nin)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(din.p, src, nin, cudaMemcpyHostToDevice, s.stream));
    if (channels == 3) {
        const size_t nout = (size_t)H * dW * 3;
        if (dout.alloc(nout)) return VSC_E_NOMEM;
        if ((rc = run_lanczos_rgb(s, (const uint8_t*)din.p, H, W, dW, (uint8_t*)dout.p))) return rc;
        CU(cudaMemcpyAsync(dst, dout.p, nout, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaStreamSynchronize(s.stream));
    } else {
        const size_t n = (size_t)H * dW;
        if (dout.alloc(n * 4)) return VSC_E_NOMEM;
        if ((rc = run_lanczos_depth(s, din.p, dtype, H, W, dW, (float*)dout.p))) return rc;
        std::vector<float> tmp(n);
        CU(cudaMemcpyAsync(tmp.data(), dout.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaStreamSynchronize(s.stream));
        if (dtype == VSC_DEPTH_U8) for (size_t i = 0; i < n; i++) ((uint8_t*)dst)[i] = (uint8_t)tmp[i];
        else if (dtype == VSC_DEPTH_U16) for (size_t i = 0; i < n; i++) ((uint16_t*)dst)[i] = (uint16_t)tmp[i];
        else memcpy(dst, tmp.data(), n * 4);
    }
    s.kH = 0;
    return VSC_OK;
}

extern "C" int vsc_stage_depth(vsc_ctx* ctx, const float* depth_st, int H, int SW, int Hs, int Ws, const vsc_params* p, float* depth_ss) {
    STAGE_BEGIN();
    if (!depth_st || !depth_ss || !p) return fail(VSC_E_INVALID, "null buffer");
    vsc_geom g = stage_geom(H, SW, SW, Hs, Ws);
    if (p->edge_softness > 0) {
        int k = ((int)(p->edge_softness * 6)) | 1; k = k < 31 ? k : 31; g.blur_k = k > 5 ? k : 5;
        if (g.blur_k / 2 >= Hs || g.blur_k / 2 >= Ws) return fail(VSC_E_PARAMS, "blur kernel does not fit");
    }
    s.kH = 0;
    int rc = ensure_tables(s, g);
    if (rc) return rc;
    const size_t n = (size_t)H * SW, ns = (size_t)Hs * Ws;
    Tmp din, dout;
    if (din.alloc(n * 4) || dout.alloc(ns * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(din.p, depth_st, n * 4, cudaMemcpyHostToDevice, s.stream));
    // min/max of the given stretched depth (the fused Lanczos kernel normally provides it)
    {
        std::vector<float> h(depth_st, depth_st + n);
        float mn = h[0], mx = h[0];
        for (size_t i = 1; i < n; i++) { mn = h[i] < mn ? h[i] : mn; mx = h[i] > mx ? h[i] : mx; }
        FrameScalars fs;
        memset(&fs, 0, sizeof fs);
        unsigned bmn, bmx;
        memcpy(&bmn, &mn, 4); memcpy(&bmx, &mx, 4);
        fs.depth_min_ord = (bmn & 0x80000000u) ? ~bmn : (bmn | 0x80000000u);
        fs.depth_max_ord = (bmx & 0x80000000u) ? ~bmx : (bmx | 0x80000000u);
        CU(cudaMemcpyAsync(s.scalars.p, &fs, sizeof fs, cudaMemcpyHostToDevice, s.stream));
        CU(cudaStreamSynchronize(s.stream));
    }
    if ((rc = run_depth_front(ctx, s, g, *p, (float*)din.p, (float*)dout.p))) return rc;
    CU(cudaMemcpyAsync(depth_ss, dout.p, ns * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    s.kH = 0;
    return VSC_OK;
}

static void unpack_view(const std::vector<uchar4>& v, uint8_t* rgb, uint8_t* mask) {
    for (size_t i = 0; i < v.size(); i++) {
        if (rgb) { rgb[3 * i] = v[i].x; rgb[3 * i + 1] = v[i].y; rgb[3 * i + 2] = v[i].z; }
        if (mask) mask[i] = v[i].w;
    }
}

extern "C" int vsc_stage_warp(vsc_ctx* ctx, const uint8_t* rgb_st, const float* depth_ss, int H, int SW, int Hs, int Ws,
                              double max_disparity, int scale255, uint8_t* left, uint8_t* left_mask, uint8_t* right,
                              uint8_t* right_mask, float* view_max) {
    STAGE_BEGIN();
    if (!rgb_st || !depth_ss) return fail(VSC_E_INVALID, "null buffer");
    vsc_geom g = stage_geom(H, SW, SW, Hs, Ws);
    s.kH = 0;
    int rc = ensure_tables(s, g);
    if (rc) return rc;
    const size_t nr = (size_t)H * SW * 3, ns = (size_t)Hs * Ws;
    Tmp drgb, dd, v0, v1;
    if (drgb.alloc(nr) || dd.alloc(ns * 4) || v0.alloc(ns * 4) || v1.alloc(ns * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(drgb.p, rgb_st, nr, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemcpyAsync(dd.p, depth_ss, ns * 4, cudaMemcpyHostToDevice, s.stream));
    if ((rc = run_warp(s, g, max_disparity, (const uint8_t*)drgb.p, (const float*)dd.p, (uchar4*)v0.p, (uchar4*)v1.p, nullptr, nullptr, nullptr, nullptr, 0))) return rc;
    if (scale255 && (rc = run_warp(s, g, max_disparity, (const uint8_t*)drgb.p, (const float*)dd.p, (uchar4*)v0.p, (uchar4*)v1.p, nullptr, nullptr, nullptr, nullptr, 2))) return rc;
    std::vector<uchar4> h0(ns), h1(ns);
    FrameScalars fs;
    CU(cudaMemcpyAsync(h0.data(), v0.p, ns * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(h1.data(), v1.p, ns * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(&fs, s.scalars.p, sizeof fs, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    unpack_view(h0, left, left_mask);
    unpack_view(h1, right, right_mask);
    if (view_max) { memcpy(&view_max[0], &fs.view_max[0], 4); memcpy(&view_max[1], &fs.view_max[1], 4); }
    s.kH = 0;
    return VSC_OK;
}

static int upload_view(Slot& s, const uint8_t* img, const uint8_t* alpha, size_t n, Tmp& d) {
    std::vector<uchar4> h(n);
    for (size_t i = 0; i < n; i++) h[i] = make_uchar4(img[3 * i], img[3 * i + 1], img[3 * i + 2], alpha ? alpha[i] : 1);
    if (d.alloc(n * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(d.p, h.data(), n * 4, cudaMemcpyHostToDevice, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return VSC_OK;
}
static int download_view(Slot& s, const Tmp& d, size_t n, uint8_t* img) {
    std::vector<uchar4> h(n);
    CU(cudaMemcpyAsync(h.data(), d.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    unpack_view(h, img, nullptr);
    return VSC_OK;
}

extern "C" int vsc_stage_bilateral(vsc_ctx* ctx, const uint8_t* img, int H, int W, double smoothing, uint8_t* out) {
    STAGE_BEGIN();
    if (!img || !out || !(smoothing > 0)) return fail(VSC_E_INVALID, "bad argument");
    const size_t n = (size_t)H * W;
    Tmp din, dout;
    int rc = upload_view(s, img, nullptr, n, din);
    if (rc) return rc;
    if (dout.alloc(n * 4)) return VSC_E_NOMEM;
    if ((rc = run_bilateral(ctx, s, H, W, smoothing, (const uchar4*)din.p, (const uchar4*)din.p, (uchar4*)dout.p, (uchar4*)dout.p, 1))) return rc;
    return download_view(s, dout, n, out);
}

extern "C" int vsc_stage_inpaint(vsc_ctx* ctx, uint8_t* img, const uint8_t* valid, int H, int W, int keep_x0, int keep_w) {
    STAGE_BEGIN();
    if (!img || !valid) return fail(VSC_E_INVALID, "null buffer");
    const size_t n = (size_t)H * W;
    Tmp dimg, dval;
    int rc = upload_view(s, img, valid, n, dimg);
    if (rc) return rc;
    Tmp dbits;
    const int wb = (W + 31) / 32;
    if (dval.alloc(n) || dbits.alloc((size_t)H * wb * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(dval.p, valid, n, cudaMemcpyHostToDevice, s.stream));
    pack_holes_kernel<<<ctx->sm_count * 8, kThreads, 0, s.stream>>>((const uint8_t*)dval.p, H, W, wb, (unsigned*)dbits.p);
    for (int attempt = 0; attempt < 4; attempt++) {
        frame_init_kernel<<<1, 32, 0, s.stream>>>(s.scalars.as<FrameScalars>());
        ViewSpec one{&s, 0, (uchar4*)dimg.p, (const unsigned*)dbits.p, keep_x0, keep_x0 + keep_w};
        if ((rc = run_telea(ctx, s, H, W, &one, 1))) return rc;
        CU(cudaMemcpyAsync(s.h_scalars, s.scalars.p, sizeof(FrameScalars), cudaMemcpyDeviceToHost, s.stream));
        CU(cudaStreamSynchronize(s.stream));
        if (!s.h_scalars->overflow) break;
        if (s.h_scalars->overflow == 0x7fffffff)
            return fail(VSC_E_STATE, "internal invariant of the hole-filling march violated (bucket range); please report the frame");
        s.qcap = (size_t)s.h_scalars->overflow * 5 / 4 + 1024;
    }
    if (s.h_scalars->overflow) return fail(VSC_E_NOMEM, "hole-filling scratch overflow persisted");
    return download_view(s, dimg, n, img);
}

extern "C" int vsc_stage_backend(vsc_ctx* ctx, const uint8_t* left, const uint8_t* right, int Hs, int Ws, int left_crop,
                                 int right_crop, int crop_w, int H, int W, double sharpen, uint8_t* out_sbs) {
    STAGE_BEGIN();
    if (!left || !right || !out_sbs) return fail(VSC_E_INVALID, "null buffer");
    if (left_crop < 0 || right_crop < 0 || left_crop + crop_w > Ws || right_crop + crop_w > Ws || crop_w < 3 || Hs < 3)
        return fail(VSC_E_PARAMS, "invalid crop window");
    vsc_geom g = stage_geom(H, W, W, Hs, Ws);
    g.left_crop = left_crop; g.right_crop = right_crop; g.crop_w = crop_w;
    const size_t n = (size_t)Hs * Ws, nout = (size_t)H * 2 * W * 3;
    Tmp d0, d1, dout;
    int rc = upload_view(s, left, nullptr, n, d0);
    if (!rc) rc = upload_view(s, right, nullptr, n, d1);
    if (rc) return rc;
    if (dout.alloc(nout)) return VSC_E_NOMEM;
    if ((rc = run_backend(s, g, sharpen, (const uchar4*)d0.p, (const uchar4*)d1.p, (uint8_t*)dout.p, VSC_LAYOUT_SBS))) return rc;
    CU(cudaMemcpyAsync(out_sbs, dout.p, nout, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return VSC_OK;
}

extern "C" int vsc_stage_normalize_f32(vsc_ctx* ctx, const float* in, size_t n, float* out) {
    STAGE_BEGIN();
    if (!in || !out || n == 0) return fail(VSC_E_INVALID, "bad argument");
    Tmp d;
    if (d.alloc(n * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(d.p, in, n * 4, cudaMemcpyHostToDevice, s.stream));
    minmax_kernel<<<ctx->sm_count * 4, kThreads, 0, s.stream>>>((const float*)d.p, n, s.scalars.as<FrameScalars>());
    normalize_kernel<<<ctx->sm_count * 4, kThreads, 0, s.stream>>>((float*)d.p, n, s.scalars.as<FrameScalars>());
    CU(cudaMemcpyAsync(out, d.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return VSC_OK;
}
extern "C" int vsc_stage_gamma_f32(vsc_ctx* ctx, const float* in, size_t n, double gamma, float* out) {
    STAGE_BEGIN();
    if (!in || !out || n == 0) return fail(VSC_E_INVALID, "bad argument");
    Tmp d, o;
    if (d.alloc(n * 4) || o.alloc(n * 4)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(d.p, in, n * 4, cudaMemcpyHostToDevice, s.stream));
    gamma_kernel<<<ctx->sm_count * 4, kThreads, 0, s.stream>>>((const float*)d.p, n, (float)gamma, ctx->pow_tab.as<double>(), (float*)o.p);
    CU(cudaMemcpyAsync(out, o.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return VSC_OK;
}
extern "C" int vsc_stage_warp_f32(vsc_ctx* ctx, const float* image, const float* depth, int C, int H, int W, double md,
                                  float* left, float* left_mask, float* right, float* right_mask) {
    STAGE_BEGIN();
    if (!image || !depth || !left || !left_mask || !right || !right_mask || C < 1 || H < 1 || W < 1)
        return fail(VSC_E_INVALID, "bad argument");
    const size_t n = (size_t)H * W;
    Tmp di, dd, o0, o1, m0, m1;
    if (di.alloc(n * C * 4) || dd.alloc(n * 4) || o0.alloc(n * C * 4) || o1.alloc(n * C * 4) || m0.alloc(n * 4) || m1.alloc(n * 4))
        return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(di.p, image, n * C * 4, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemcpyAsync(dd.p, depth, n * 4, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemsetAsync(o0.p, 0, n * C * 4, s.stream)); CU(cudaMemsetAsync(o1.p, 0, n * C * 4, s.stream));
    CU(cudaMemsetAsync(m0.p, 0, n * 4, s.stream)); CU(cudaMemsetAsync(m1.p, 0, n * 4, s.stream));
    // the depth's extremes bound how far a source moves, i.e. the halo each segment scans (the depth may be unnormalised)
    minmax_kernel<<<ctx->sm_count * 4, kThreads, 0, s.stream>>>((const float*)dd.p, n, s.scalars.as<FrameScalars>());
    const int nseg = (W + 1023) / 1024;
    const int TS = (int)align_up((size_t)(W + nseg - 1) / nseg, 32);
    dim3 grid(nseg, H);
    warp_f32_kernel<<<grid, kThreads, (size_t)TS * 16, s.stream>>>((const float*)di.p, (const float*)dd.p, C, H, W, (float)md,
                                                                  s.scalars.as<FrameScalars>(), TS, (float*)o0.p, (float*)m0.p,
                                                                  (float*)o1.p, (float*)m1.p);
    KCHECK(s);
    CU(cudaMemcpyAsync(left, o0.p, n * C * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(right, o1.p, n * C * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(left_mask, m0.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(right_mask, m1.p, n * 4, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return VSC_OK;
}

// ---- depth-map post-processing (depth_map_generator.py:217-236): resize + normalise + quantise ---------------------
static int enqueue_depth_post(vsc_ctx* ctx, Slot& s, cudaStream_t stream, const float* d_src, int h, int w, int H, int W, int bits, void* d_dst) {
    if (s.dp_scalars.ensure(sizeof(DepthPostScalars))) return VSC_E_NOMEM;
    DepthPostScalars* sc = s.dp_scalars.as<DepthPostScalars>();
    const double sx = 1.0 / ((double)W / (double)w), sy = 1.0 / ((double)H / (double)h);
    dim3 grid((W + kThreads - 1) / kThreads, H);
    depth_post_init_kernel<<<1, 1, 0, stream>>>(sc);
    if (bits == 16) {
        depth_post_kernel<0, uint16_t><<<grid, kThreads, 0, stream>>>(d_src, h, w, H, W, sx, sy, sc, (uint16_t*)d_dst, 65535.f);
        depth_post_kernel<1, uint16_t><<<grid, kThreads, 0, stream>>>(d_src, h, w, H, W, sx, sy, sc, (uint16_t*)d_dst, 65535.f);
    } else {
        depth_post_kernel<0, uint8_t><<<grid, kThreads, 0, stream>>>(d_src, h, w, H, W, sx, sy, sc, (uint8_t*)d_dst, 255.f);
        depth_post_kernel<1, uint8_t><<<grid, kThreads, 0, stream>>>(d_src, h, w, H, W, sx, sy, sc, (uint8_t*)d_dst, 255.f);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(VSC_E_CUDA, "depth post-processing launch failed: %s", cudaGetErrorString(e));
    (void)ctx;
    return VSC_OK;
}
static int depth_post_args_ok(const void* a, const void* b, int h, int w, int H, int W, int bits) {
    if (!a || !b) return fail(VSC_E_INVALID, "null buffer");
    if (h < 1 || w < 1 || H < 1 || W < 1 || (bits != 8 && bits != 16)) return fail(VSC_E_INVALID, "bad depth post-processing geometry / bit depth");
    return VSC_OK;
}
extern "C" int vsc_depth_post_device(vsc_ctx* ctx, int slot, const float* d_depth, int h, int w, int H, int W, int bits, void* d_out) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr) return fail(VSC_E_INVALID, "bad context or slot");
    int rc = depth_post_args_ok(d_depth, d_out, h, w, H, W, bits);
    if (rc) return rc;
    if (fr->busy) return fail(VSC_E_STATE, "slot %d still has frames in flight; call vsc_wait first", slot);
    CU(cudaSetDevice(ctx->device));
    return enqueue_depth_post(ctx, *fr, fr->stream, d_depth, h, w, H, W, bits, d_out);
}
extern "C" int vsc_stage_png(vsc_ctx* ctx, const uint8_t* rgb, int H, int W, uint8_t* out, size_t capacity, size_t* bytes) {
    STAGE_BEGIN();
    if (!rgb || !out || !bytes || H < 1 || W < 1) return fail(VSC_E_INVALID, "bad argument");
    if ((long long)W * 3 + 1 > (1ll << 31) - 1) return fail(VSC_E_INVALID, "frame width %d too large for PNG output", W);
    const size_t cap = png_capacity(H, W), nin = (size_t)H * W * 3;
    if (capacity < cap) return fail(VSC_E_INVALID, "output capacity %zu is below vsc_encoded_capacity (%zu)", capacity, cap);
    Tmp din, dout;
    if (din.alloc(nin) || dout.alloc(cap) || s.png_stats.ensure(3 * sizeof(unsigned long long))) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(din.p, rgb, nin, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemsetAsync(s.png_stats.p, 0, 3 * sizeof(unsigned long long), s.stream));
    s.l_out = (uint8_t*)din.p;
    s.l_png = (uint8_t*)dout.p;
    int rc = run_png(s, &s, 1, H, W, s.png_stats.as<unsigned long long>());
    if (rc) { cudaStreamSynchronize(s.stream); return rc; }
    CU(cudaStreamSynchronize(s.stream));
    *bytes = (size_t)*s.h_png;
    CU(cudaMemcpyAsync(out, dout.p, *bytes, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    s.l_out = nullptr;
    s.l_png = nullptr;
    return VSC_OK;
}
extern "C" int vsc_debug_png_stats(vsc_ctx* ctx, unsigned long long* out) {
    if (!ctx || !out) return fail(VSC_E_INVALID, "bad argument");
    Slot& s = ctx->slots[0];
    if (!s.png_stats.p) return fail(VSC_E_STATE, "no vsc_stage_png call on this context yet");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpy(out, s.png_stats.p, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return VSC_OK;
}

extern "C" int vsc_stage_depth_post(vsc_ctx* ctx, const float* depth, int h, int w, int H, int W, int bits, void* out, int* ok) {
    STAGE_BEGIN();
    int rc = depth_post_args_ok(depth, out, h, w, H, W, bits);
    if (rc) return rc;
    const size_t nin = (size_t)h * w * 4, nout = (size_t)H * W * (bits == 16 ? 2 : 1);
    Tmp din, dout;
    if (din.alloc(nin) || dout.alloc(nout)) return VSC_E_NOMEM;
    CU(cudaMemcpyAsync(din.p, depth, nin, cudaMemcpyHostToDevice, s.stream));
    if ((rc = enqueue_depth_post(ctx, s, s.stream, (const float*)din.p, h, w, H, W, bits, dout.p))) return rc;
    DepthPostScalars sc;
    CU(cudaMemcpyAsync(out, dout.p, nout, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(&sc, s.dp_scalars.p, sizeof sc, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    if (ok) *ok = ord2f(sc.max_ord) - ord2f(sc.min_ord) > 0.f;     // flat map: the reference writes no depth file
    return VSC_OK;
}

// debug: copy the Telea state of slot 0 (after vsc_stage_inpaint) to the host
extern "C" int vsc_debug_telea_state(vsc_ctx* ctx, int view, float* tt, uint8_t* st, uint32_t* ord, size_t n) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    Slot& s = ctx->slots[0];
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    if (tt) CU(cudaMemcpy(tt, s.tt[view].p, n * 4, cudaMemcpyDeviceToHost));
    if (st) CU(cudaMemcpy(st, s.st[view].p, n, cudaMemcpyDeviceToHost));
    if (ord) CU(cudaMemcpy(ord, s.pstate[view].p, n * 4, cudaMemcpyDeviceToHost));
    return VSC_OK;
}

// debug: copy an intermediate buffer of slot 0 (after a completed frame) to the host.
// which: 0 rgb_st, 1 depth_st (normalised), 2 depth_ss, 3/4 viewA L/R, 5/6 viewB L/R, 7/8 hole bitmaps L/R
extern "C" int vsc_debug_fetch(vsc_ctx* ctx, int which, void* dst, size_t bytes) {
    if (!ctx || !dst) return fail(VSC_E_INVALID, "null argument");
    Slot& s = ctx->slots[0];
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    DevBuf* b[] = {&s.rgb_st, &s.depth_st, &s.depth_ss, &s.viewA[0], &s.viewA[1], &s.viewB[0], &s.viewB[1], &s.vmask[0], &s.vmask[1]};
    if (which < 0 || which > 8 || !b[which]->p || b[which]->cap < bytes) return fail(VSC_E_INVALID, "bad buffer id or size");
    CU(cudaMemcpy(dst, b[which]->p, bytes, cudaMemcpyDeviceToHost));
    return VSC_OK;
}

// which = 0: rcp_rn_1_256 against __frcp_rn on [1, 256); which = 1: div3_exact / div3_exact2 against __fdiv_rn(x, 3)
// on [0, 2295 + 16 ulp].  *mismatches = number of floats of the range where they differ (must be 0).
extern "C" int vsc_debug_selftest(vsc_ctx* ctx, int which, unsigned long long* mismatches) {
    if (!ctx || !mismatches || which < 0 || which > 1) return fail(VSC_E_INVALID, "bad argument");
    CU(cudaSetDevice(ctx->device));
    unsigned long long* d_bad = nullptr;
    CU(cudaMalloc(&d_bad, sizeof *d_bad));
    cudaError_t e = cudaMemset(d_bad, 0, sizeof *d_bad);
    if (e == cudaSuccess) {
        const float top = 2295.0f;
        unsigned tb;
        memcpy(&tb, &top, 4);
        const unsigned lo = which == 0 ? 0x3f800000u : 0u, hi = which == 0 ? 0x437fffffu : tb + 16u;
        selftest_kernel<<<ctx->sm_count * 8, kThreads>>>(which, lo, hi, d_bad);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpy(mismatches, d_bad, sizeof *d_bad, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_bad);
    if (e != cudaSuccess) return fail(VSC_E_CUDA, "selftest: %s", cudaGetErrorString(e));
    return VSC_OK;
}

// ------------------------------------------------------------------------------------------------
// measurement helpers
// ------------------------------------------------------------------------------------------------
extern "C" int vsc_set_profiling(vsc_ctx* ctx, int on) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    ctx->profiling = on != 0;
    for (auto& s : ctx->slots) s.prof = ctx->profiling;
    return VSC_OK;
}
// per-kernel device times of the last completed frame on `slot` (needs vsc_set_profiling(ctx,1) before submit)
extern "C" int vsc_slot_kernel_times(vsc_ctx* ctx, int slot, int max_n, const char** names, float* ms) {
    Slot* fr = group_lead(ctx, slot);
    if (!fr || !names || !ms) return fail(VSC_E_INVALID, "bad argument");
    int n = 0;
    for (int f = 0; f < ctx->group_size; f++) {
        Slot& s = fr[f];
        for (int i = 0; i < s.pcount && n < max_n; i++, n++) {
            names[n] = s.pname[i];
            if (cudaEventElapsedTime(&ms[n], s.pev[2 * i], s.pev[2 * i + 1]) != cudaSuccess) ms[n] = -1.f;
        }
    }
    return n;
}
// device-side timer spanning all slot streams: begin makes every slot stream wait on a start event,
// end records after every slot stream has drained; elapsed is measured between the two events.
extern "C" int vsc_timer_begin(vsc_ctx* ctx) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    CU(cudaSetDevice(ctx->device));
    if (!ctx->tstream) {
        CU(cudaStreamCreateWithFlags(&ctx->tstream, cudaStreamNonBlocking));
        CU(cudaEventCreate(&ctx->t0)); CU(cudaEventCreate(&ctx->t1));
        ctx->tslot.resize(ctx->slots.size());
        for (auto& e : ctx->tslot) CU(cudaEventCreate(&e));
    }
    CU(cudaDeviceSynchronize());
    CU(cudaEventRecord(ctx->t0, ctx->tstream));
    for (auto& s : ctx->slots) if (s.owns_stream) CU(cudaStreamWaitEvent(s.stream, ctx->t0, 0));
    return VSC_OK;
}
extern "C" int vsc_timer_end(vsc_ctx* ctx, float* ms) {
    if (!ctx || !ms || !ctx->tstream) return fail(VSC_E_INVALID, "timer not started");
    CU(cudaSetDevice(ctx->device));
    for (size_t i = 0; i < ctx->slots.size(); i++) {
        if (!ctx->slots[i].owns_stream) continue;
        CU(cudaEventRecord(ctx->tslot[i], ctx->slots[i].stream));
        CU(cudaStreamWaitEvent(ctx->tstream, ctx->tslot[i], 0));
    }
    CU(cudaEventRecord(ctx->t1, ctx->tstream));
    CU(cudaEventSynchronize(ctx->t1));
    CU(cudaEventElapsedTime(ms, ctx->t0, ctx->t1));
    return VSC_OK;
}

// debug: Telea phase counters of slot 0 (all zero unless built with -DVSC_TELEA_STATS)
extern "C" int vsc_debug_telea_stats(vsc_ctx* ctx, unsigned long long* out64) {
    if (!ctx || !out64) return fail(VSC_E_INVALID, "null argument");
    Slot& s = ctx->slots[0];
    memset(out64, 0, 64 * 8);
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    if (s.tstats.p) CU(cudaMemcpy(out64, s.tstats.p, 64 * 8, cudaMemcpyDeviceToHost));
    return VSC_OK;
}

// test hook: shrink the hole-filling queue scratch of every slot so that the overflow -> regrow -> re-run path
// (vsc_wait / vsc_stage_inpaint) can be exercised
extern "C" int vsc_debug_set_telea_capacity(vsc_ctx* ctx, size_t entries) {
    if (!ctx) return fail(VSC_E_INVALID, "null context");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    for (auto& s : ctx->slots) {
        if (s.busy) return fail(VSC_E_STATE, "a slot is busy");
        for (int v = 0; v < 2; v++) { s.qkey[v].release(); s.qidx[v].release(); }
        s.qcap = entries;
    }
    return VSC_OK;
}
