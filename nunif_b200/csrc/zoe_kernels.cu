// Non-GEMM kernels of the ZoeD_N metric depth network (BEiT-L/16 encoder + MiDaS DPT head + ZoeDepth bins head) that
// Depth-Anything does not already provide (depth_kernels.cu: add+LayerNorm, flash attention, relu/upsample/im2col helpers).
// The reference runs the network under fp16 autocast (iw3/zoedepth_model.py:23-27): convs / Linears in fp16 with fp32
// accumulate, softplus / log / softmax / interpolate-of-fp32 in fp32 - mirrored here: everything that feeds a GEMM is
// fp16 NHWC, the bin centres and the final log-binomial mixture are fp32.
// Restated architecture: oracle/zoedepth.py (MiDaS backbones/beit.py, dpt_depth.py; ZoeDepth zoedepth_v1.py, attractor.py,
// dist_layers.py, localbins_layers.py).
#include "zoe_kernels.h"

namespace nb200 {

namespace {
constexpr int PATCH = 16;
constexpr int NBINS = 64;
constexpr float LOG2E = 1.4426950408889634f;

// F.softplus (beta 1, threshold 20)
__device__ __forceinline__ float softplus(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// ATen upsample_bilinear2d align_corners=True source index: src = dst * (in - 1) / (out - 1)
struct Lerp {
    int i0, i1;
    float l0, l1;
};
__device__ __forceinline__ Lerp lerp_ac(int dst, float scale, int in) {
    const float f = __fmul_rn(scale, (float)dst);
    Lerp r;
    r.i0 = min((int)f, in - 1);
    r.i1 = min(r.i0 + 1, in - 1);
    r.l1 = f - (float)r.i0;
    r.l0 = 1.f - r.l1;
    return r;
}
inline float ac_scale(int in, int out) { return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f; }
}  // namespace

// ------------------------------------------------------------------------------------------ encoder edges
__global__ void __launch_bounds__(256) zoe_patch_im2col_kernel(const float* __restrict__ x, __half* __restrict__ A, int B, int H, int W,
                                                                int ph, int pw) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    constexpr int K = 3 * PATCH * PATCH;
    const long long total = (long long)B * ph * pw * K;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int k = (int)(i % K);
    const long long row = i / K;
    const int kx = k % PATCH, ky = (k / PATCH) % PATCH, c = k / (PATCH * PATCH);
    const int px = (int)(row % pw), py = (int)((row / pw) % ph), b = (int)(row / ((long long)pw * ph));
    A[i] = __float2half_rn(__ldg(x + (((size_t)b * 3 + c) * H + py * PATCH + ky) * W + px * PATCH + kx));
}

__global__ void __launch_bounds__(256) zoe_assemble_tokens_kernel(const __half* __restrict__ T, const float* __restrict__ cls,
                                                                   float* __restrict__ X, int B, int P, int dim) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * (P + 1) * dim;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % dim);
    const long long r = i / dim;
    const int n = (int)(r % (P + 1)), b = (int)(r / (P + 1));
    X[i] = n == 0 ? cls[c] : __half2float(T[((size_t)b * P + (n - 1)) * dim + c]);
}

__global__ void __launch_bounds__(256) zoe_add_cast_kernel(float4* __restrict__ X, const uint2* __restrict__ delta, uint2* __restrict__ out,
                                                            long long n4) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float4 v = X[i];
    if (delta) {
        const uint2 raw = delta[i];
        const __half2* h = reinterpret_cast<const __half2*>(&raw);
        const float2 d0 = __half22float2(h[0]), d1 = __half22float2(h[1]);
        v.x += d0.x; v.y += d0.y; v.z += d1.x; v.w += d1.y;
        X[i] = v;
    }
    __align__(8) __half2 o[2];
    o[0] = __floats2half2_rn(v.x, v.y);
    o[1] = __floats2half2_rn(v.z, v.w);
    out[i] = *reinterpret_cast<const uint2*>(o);
}

// one thread per (head, q, k): index arithmetic of gen_relative_position_index, no index tensor
__global__ void __launch_bounds__(256) zoe_expand_rel_bias_kernel(const float* __restrict__ table, int ph, int pw, int heads,
                                                                   float* __restrict__ bias, int ldb) {
    const int N = ph * pw + 1;
    const long long total = (long long)heads * N * N;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int k = (int)(i % N);
    const long long r = i / N;
    const int q = (int)(r % N), h = (int)(r / N);
    const int nrd = (2 * ph - 1) * (2 * pw - 1) + 3;
    int idx;
    if (q == 0 && k == 0) idx = nrd - 1;
    else if (q == 0) idx = nrd - 3;
    else if (k == 0) idx = nrd - 2;
    else {
        const int qy = (q - 1) / pw, qx = (q - 1) % pw, ky = (k - 1) / pw, kx = (k - 1) % pw;
        idx = (qy - ky + ph - 1) * (2 * pw - 1) + (qx - kx + pw - 1);
    }
    bias[((size_t)h * N + q) * ldb + k] = table[(size_t)idx * heads + h] * LOG2E;
}

__global__ void __launch_bounds__(256) zoe_readout_concat_kernel(const uint4* __restrict__ F, int B, int P, int dim8, uint4* __restrict__ A) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * P * 2 * dim8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % (2 * dim8));
    const long long row = i / (2 * dim8);
    const int n = (int)(row % P), b = (int)(row / P);
    const size_t src = c < dim8 ? ((size_t)b * (P + 1) + 1 + n) * dim8 + c : ((size_t)b * (P + 1)) * dim8 + (c - dim8);
    A[i] = __ldg(F + src);
}

// ------------------------------------------------------------------------------------------ bins head
__global__ void __launch_bounds__(256) zoe_add_upsampled_kernel(const __half* __restrict__ e, const __half* __restrict__ prev, int B, int h,
                                                                 int w, int C8, int H, int W, float sy, float sx, __half* __restrict__ y) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * H * W * C8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c8 = (int)(i % C8);
    long long r = i / C8;
    const int X = (int)(r % W);
    r /= W;
    const int Y = (int)(r % H), b = (int)(r / H);
    const Lerp ly = lerp_ac(Y, sy, h), lx = lerp_ac(X, sx, w);
    const size_t C = (size_t)C8 * 8;
    const __half* p = prev + (size_t)b * h * w * C + (size_t)c8 * 8;
    const uint4 v00 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i0 * w + lx.i0) * C));
    const uint4 v01 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i0 * w + lx.i1) * C));
    const uint4 v10 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i1 * w + lx.i0) * C));
    const uint4 v11 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i1 * w + lx.i1) * C));
    const uint4 ve = __ldg(reinterpret_cast<const uint4*>(e + (size_t)i * 8));
    const __half2 *a = reinterpret_cast<const __half2*>(&v00), *bq = reinterpret_cast<const __half2*>(&v01);
    const __half2 *c = reinterpret_cast<const __half2*>(&v10), *d = reinterpret_cast<const __half2*>(&v11);
    const __half2* ee = reinterpret_cast<const __half2*>(&ve);
    __align__(16) __half2 o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 fa = __half22float2(a[k]), fb = __half22float2(bq[k]), fc = __half22float2(c[k]), fd = __half22float2(d[k]);
        // the interpolated embedding is an fp16 tensor in the reference (interpolate of an fp16 conv output), then fp16 + fp16
        const __half2 up = __floats2half2_rn(ly.l0 * (lx.l0 * fa.x + lx.l1 * fb.x) + ly.l1 * (lx.l0 * fc.x + lx.l1 * fd.x),
                                             ly.l0 * (lx.l0 * fa.y + lx.l1 * fb.y) + ly.l1 * (lx.l0 * fc.y + lx.l1 * fd.y));
        const float2 fu = __half22float2(up), fe = __half22float2(ee[k]);
        o[k] = __floats2half2_rn(fe.x + fu.x, fe.y + fu.y);
    }
    *reinterpret_cast<uint4*>(y + (size_t)i * 8) = *reinterpret_cast<const uint4*>(o);
}

__global__ void __launch_bounds__(256) zoe_softplus_kernel(const __half* __restrict__ x, float* __restrict__ out, long long n) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = softplus(__half2float(x[i]));
}

// one thread per (pixel, bin): 64 consecutive threads share a pixel, so the prev_bin gathers are coalesced 256-byte rows
__global__ void __launch_bounds__(256) zoe_attractor_kernel(const __half* __restrict__ apre, int lda, int na, const float* __restrict__ prev,
                                                             int B, int h, int w, int H, int W, float sy, float sx, float* __restrict__ out) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * H * W * NBINS;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int k = (int)(i % NBINS);
    long long pix = i / NBINS;
    const int X = (int)(pix % W);
    long long r = pix / W;
    const int Y = (int)(r % H), b = (int)(r / H);
    const Lerp ly = lerp_ac(Y, sy, h), lx = lerp_ac(X, sx, w);
    const float* p = prev + (size_t)b * h * w * NBINS + k;
    const float c00 = __ldg(p + ((size_t)ly.i0 * w + lx.i0) * NBINS), c01 = __ldg(p + ((size_t)ly.i0 * w + lx.i1) * NBINS);
    const float c10 = __ldg(p + ((size_t)ly.i1 * w + lx.i0) * NBINS), c11 = __ldg(p + ((size_t)ly.i1 * w + lx.i1) * NBINS);
    const float c = ly.l0 * (lx.l0 * c00 + lx.l1 * c01) + ly.l1 * (lx.l0 * c10 + lx.l1 * c11);
    const __half* ap = apre + (size_t)pix * lda;
    float delta = 0.f;
    for (int j = 0; j < na; ++j) {
        const float dx = softplus(__half2float(__ldg(ap + j))) - c;
        delta += dx / (1.f + 300.f * dx * dx);     // inv_attractor with its default alpha = 300, gamma = 2 (upstream quirk)
    }
    out[i] = c + delta / (float)na;
}

// one thread per (pixel, group of 8 channels): groups 0..15 = the resampled embedding, 16..19 = the activation, 20 = relative
// depth + zeros, 21..23 = zeros (channel order chosen at pack time, zoe_model.inl)
__global__ void __launch_bounds__(256) zoe_clb_concat_kernel(const __half* __restrict__ act, const float* __restrict__ rel,
                                                              const __half* __restrict__ emb, int B, int h, int w, int H, int W, float sy,
                                                              float sx, __half* __restrict__ A) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    constexpr int G = 24;
    const long long total = (long long)B * H * W * G;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int g = (int)(i % G);
    const long long pix = i / G;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (g < 16) {
        const int X = (int)(pix % W);
        const long long r = pix / W;
        const int Y = (int)(r % H), b = (int)(r / H);
        const Lerp ly = lerp_ac(Y, sy, h), lx = lerp_ac(X, sx, w);
        const __half* p = emb + (size_t)b * h * w * 128 + g * 8;
        const uint4 v00 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i0 * w + lx.i0) * 128));
        const uint4 v01 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i0 * w + lx.i1) * 128));
        const uint4 v10 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i1 * w + lx.i0) * 128));
        const uint4 v11 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)ly.i1 * w + lx.i1) * 128));
        const __half2 *a = reinterpret_cast<const __half2*>(&v00), *bq = reinterpret_cast<const __half2*>(&v01);
        const __half2 *c = reinterpret_cast<const __half2*>(&v10), *d = reinterpret_cast<const __half2*>(&v11);
        __half2* o = reinterpret_cast<__half2*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fa = __half22float2(a[k]), fb = __half22float2(bq[k]), fc = __half22float2(c[k]), fd = __half22float2(d[k]);
            o[k] = __floats2half2_rn(ly.l0 * (lx.l0 * fa.x + lx.l1 * fb.x) + ly.l1 * (lx.l0 * fc.x + lx.l1 * fd.x),
                                     ly.l0 * (lx.l0 * fa.y + lx.l1 * fb.y) + ly.l1 * (lx.l0 * fc.y + lx.l1 * fd.y));
        }
    } else if (g < 20) {
        v = __ldg(reinterpret_cast<const uint4*>(act + (size_t)pix * 32 + (g - 16) * 8));
    } else if (g == 20) {
        v.x = (uint32_t)__half_as_ushort(__float2half_rn(__ldg(rel + pix)));
    }
    *reinterpret_cast<uint4*>(A + (size_t)i * 8) = v;
}

// one warp per pixel: lanes split the 80-wide dot products, then each lane owns bins k = lane and lane + 32
__global__ void __launch_bounds__(256) zoe_clb_final_kernel(const __half* __restrict__ g, int ldg, const float* __restrict__ w2, const float* __restrict__ b2,
                                                             const float* __restrict__ bins, int B, int h, int w, int H, int W, float sy,
                                                             float sx, float* __restrict__ depth) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    __shared__ float sw[4 * 80 + 4];
    __shared__ float slb[NBINS];
    for (int t = threadIdx.x; t < 4 * 80 + 4; t += blockDim.x) sw[t] = t < 320 ? w2[t] : b2[t - 320];
    if (threadIdx.x < NBINS) {
        // log_binom(n = 63, k) with Stirling's approximation and the upstream epsilons (dist_layers.py log_binom)
        const float eps = 1e-7f, n = 63.f + eps, k = (float)threadIdx.x + eps;
        slb[threadIdx.x] = n * logf(n) - k * logf(k) - (n - k) * logf(n - k + eps);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long npix = (long long)B * H * W, wstride = (long long)gridDim.x * (blockDim.x >> 5);
    // persistent warps: the weight / log-binomial tables are staged once per block, not once per 8 pixels
    for (long long pix = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); pix < npix; pix += wstride) {
    const __half* gp = g + (size_t)pix * ldg;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = lane; c < 80; c += 32) {
        const float v = __half2float(__ldg(gp + c));
#pragma unroll
        for (int o = 0; o < 4; ++o) acc[o] = fmaf(v, sw[o * 80 + c], acc[o]);
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], s);
        // (the reference's conv output is an fp16 tensor under autocast; the fp32 sum is kept here: these 4 values are
        // amplified by up to 63 / min_temp ~ 3000 in the logits below, so their rounding dominates the output error)
        acc[o] = softplus(acc[o] + sw[320 + o]) + 1e-4f;
    }
    const float p = acc[0] / (acc[0] + acc[1]);
    const float tn = acc[2] / (acc[2] + acc[3]);
    const float temp = (50.0f - 0.0212f) * tn + 0.0212f;
    const float lp = logf(fminf(fmaxf(p, 1e-4f), 1.f)), lq = logf(fminf(fmaxf(1.f - p, 1e-4f), 1.f));
    float y[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float k = (float)(lane + 32 * j);
        y[j] = (slb[lane + 32 * j] + k * lp + (63.f - k) * lq) / temp;
    }
    float mx = fmaxf(y[0], y[1]);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    const float e0 = expf(y[0] - mx), e1 = expf(y[1] - mx);
    // bin centres at this pixel
    const int X = (int)(pix % W);
    const long long r = pix / W;
    const int Y = (int)(r % H), b = (int)(r / H);
    const Lerp ly = lerp_ac(Y, sy, h), lx = lerp_ac(X, sx, w);
    const float* bp = bins + (size_t)b * h * w * NBINS;
    float num = 0.f;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int k = lane + 32 * j;
        const float c00 = __ldg(bp + ((size_t)ly.i0 * w + lx.i0) * NBINS + k), c01 = __ldg(bp + ((size_t)ly.i0 * w + lx.i1) * NBINS + k);
        const float c10 = __ldg(bp + ((size_t)ly.i1 * w + lx.i0) * NBINS + k), c11 = __ldg(bp + ((size_t)ly.i1 * w + lx.i1) * NBINS + k);
        const float c = ly.l0 * (lx.l0 * c00 + lx.l1 * c01) + ly.l1 * (lx.l0 * c10 + lx.l1 * c11);
        num = fmaf(j == 0 ? e0 : e1, c, num);
    }
    float den = e0 + e1;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        num += __shfl_xor_sync(0xffffffffu, num, s);
        den += __shfl_xor_sync(0xffffffffu, den, s);
    }
    if (lane == 0) depth[pix] = num / den;
    }
}

// ------------------------------------------------------------------------------------------ host wrappers
int zoe_patch_im2col(cudaStream_t st, const float* x, int B, int H, int W, __half* A) {
    const int ph = H / PATCH, pw = W / PATCH;
    const long long total = (long long)B * ph * pw * 3 * PATCH * PATCH;
    zoe_patch_im2col_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(x, A, B, H, W, ph, pw);
    NB_LAUNCHED();
    return 0;
}

int zoe_assemble_tokens(cudaStream_t st, const __half* T, const float* cls, float* X32, int B, int P, int dim) {
    const long long total = (long long)B * (P + 1) * dim;
    zoe_assemble_tokens_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(T, cls, X32, B, P, dim);
    NB_LAUNCHED();
    return 0;
}

int zoe_add_cast(cudaStream_t st, float* X32, const __half* delta, __half* out, long long n) {
    NB_CHECK(n % 4 == 0, "element count must be a multiple of 4");
    zoe_add_cast_kernel<<<(unsigned)cdiv64(n / 4, 256), 256, 0, st>>>(reinterpret_cast<float4*>(X32), reinterpret_cast<const uint2*>(delta),
                                                                      reinterpret_cast<uint2*>(out), n / 4);
    NB_LAUNCHED();
    return 0;
}

int zoe_expand_rel_bias(cudaStream_t st, const float* table, int ph, int pw, int heads, float* bias, int ldb) {
    const long long N = (long long)ph * pw + 1, total = (long long)heads * N * N;
    NB_CHECK(ldb >= N, "bias row stride too small");
    zoe_expand_rel_bias_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(table, ph, pw, heads, bias, ldb);
    NB_LAUNCHED();
    return 0;
}

int zoe_readout_concat(cudaStream_t st, const __half* F, int B, int P, int dim, __half* A) {
    NB_CHECK(dim % 8 == 0, "embedding dim must be a multiple of 8");
    const long long total = (long long)B * P * 2 * (dim / 8);
    zoe_readout_concat_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(reinterpret_cast<const uint4*>(F), B, P, dim / 8,
                                                                            reinterpret_cast<uint4*>(A));
    NB_LAUNCHED();
    return 0;
}

int zoe_add_upsampled(cudaStream_t st, const __half* e, const __half* prev, int B, int h, int w, int C, int H, int W, __half* y) {
    NB_CHECK(C % 8 == 0, "channels must be a multiple of 8");
    const long long total = (long long)B * H * W * (C / 8);
    zoe_add_upsampled_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(e, prev, B, h, w, C / 8, H, W, ac_scale(h, H), ac_scale(w, W), y);
    NB_LAUNCHED();
    return 0;
}

int zoe_softplus(cudaStream_t st, const __half* x, float* out, long long n) {
    zoe_softplus_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, st>>>(x, out, n);
    NB_LAUNCHED();
    return 0;
}

int zoe_attractor(cudaStream_t st, const __half* apre, int lda, int na, const float* prev_bin, int B, int h, int w, int H, int W,
                  float* out) {
    NB_CHECK(na >= 1 && na <= lda, "bad attractor count");
    const long long total = (long long)B * H * W * NBINS;
    zoe_attractor_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(apre, lda, na, prev_bin, B, h, w, H, W, ac_scale(h, H), ac_scale(w, W), out);
    NB_LAUNCHED();
    return 0;
}

int zoe_clb_concat(cudaStream_t st, const __half* act, const float* rel, const __half* emb, int B, int h, int w, int H, int W, __half* A) {
    const long long total = (long long)B * H * W * 24;
    zoe_clb_concat_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(act, rel, emb, B, h, w, H, W, ac_scale(h, H), ac_scale(w, W), A);
    NB_LAUNCHED();
    return 0;
}

int zoe_clb_final(cudaStream_t st, const __half* g, int ldg, const float* w2, const float* b2, const float* bins, int B, int h, int w, int H,
                  int W, float* depth) {
    NB_CHECK(ldg >= 80, "hidden row stride too small");
    const long long npix = (long long)B * H * W;
    const long long blocks = cdiv64(npix, 8), cap = (long long)device_sm_count() * 8;
    zoe_clb_final_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(g, ldg, w2, b2, bins, B, h, w, H, W, ac_scale(h, H), ac_scale(w, W), depth);
    NB_LAUNCHED();
    return 0;
}

}  // namespace nb200

using namespace nb200;

// Low-level ops of the depth networks exposed for unit tests (see include/nunif_b200.h).
extern "C" int nb200_zoe_expand_rel_bias(const float* table, int ph, int pw, int heads, float* bias, int ldb, void* stream) {
    NB_CHECK(table && bias, "null pointer");
    NB_CHECK(ph >= 1 && pw >= 1 && heads >= 1, "empty token grid");
    return zoe_expand_rel_bias((cudaStream_t)stream, table, ph, pw, heads, bias, ldb);
}

extern "C" int nb200_zoe_attractor(const void* apre, int lda, int na, const float* prev_bin, int B, int h, int w, int H, int W,
                                   float* out, void* stream) {
    NB_CHECK(apre && prev_bin && out, "null pointer");
    NB_CHECK(B >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, "empty image");
    return zoe_attractor((cudaStream_t)stream, (const __half*)apre, lda, na, prev_bin, B, h, w, H, W, out);
}

extern "C" int nb200_zoe_clb_final(const void* g, int ldg, const float* w2, const float* b2, const float* bins, int B, int h, int w,
                                   int H, int W, float* depth, void* stream) {
    NB_CHECK(g && w2 && b2 && bins && depth, "null pointer");
    NB_CHECK(B >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, "empty image");
    return zoe_clb_final((cudaStream_t)stream, (const __half*)g, ldg, w2, b2, bins, B, h, w, H, W, depth);
}
