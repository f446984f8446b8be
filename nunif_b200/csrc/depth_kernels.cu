// Non-GEMM kernels of the Depth-Anything-V2 network (DINOv2 ViT encoder + DPT head):
// patch im2col, token assembly, fused residual-add + LayerNorm on an fp32 residual stream, flash attention on
// mma.sync tensor cores, and the small NHWC helpers of the DPT head.  The reference runs this network under fp16
// autocast (iw3/depth_anything_model.py:113-119): Linears/convs/matmuls in fp16 with fp32 accumulate, LayerNorm and
// softmax in fp32, and the residual stream stays fp32 (cat with the fp32 cls token promotes it) - mirrored here.
// Restated architecture: oracle/depth_anything.py (upstream dinov2 vision_transformer.py, Depth-Anything-V2 dpt.py).
#include "depth_kernels.h"

namespace nb200 {

namespace {
constexpr int PATCH = 14;

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, const void* smem_row) {
    const uint32_t addr = (uint32_t)__cvta_generic_to_shared(smem_row);
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
}  // namespace

// ------------------------------------------------------------------------------------------ patch embedding
__global__ void __launch_bounds__(256) patch_im2col_kernel(const float* __restrict__ x, __half* __restrict__ A, int B, int H, int W,
                                                            int ph, int pw, int kpad) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * ph * pw * kpad;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int k = (int)(i % kpad);
    const long long row = i / kpad;
    float v = 0.f;
    if (k < 3 * PATCH * PATCH) {
        const int kx = k % PATCH, ky = (k / PATCH) % PATCH, c = k / (PATCH * PATCH);
        const int px = (int)(row % pw), py = (int)((row / pw) % ph), b = (int)(row / ((long long)pw * ph));
        v = __ldg(x + (((size_t)b * 3 + c) * H + py * PATCH + ky) * W + px * PATCH + kx);
    }
    A[i] = __float2half_rn(v);
}

__global__ void __launch_bounds__(256) assemble_tokens_kernel(const __half* __restrict__ T, const float* __restrict__ cls,
                                                               const float* __restrict__ pos, float* __restrict__ X, int B, int P,
                                                               int dim) {
    const long long total = (long long)B * (P + 1) * dim;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % dim);
    const long long r = i / dim;
    const int n = (int)(r % (P + 1)), b = (int)(r / (P + 1));
    const float v = n == 0 ? cls[c] : __half2float(T[((size_t)b * P + (n - 1)) * dim + c]);
    X[i] = v + pos[(size_t)n * dim + c];
}

// ------------------------------------------------------------------------------------------ add + LayerNorm
// one warp per row; DIM/128 float4 per lane
template <int DIM>
__global__ void __launch_bounds__(256) add_layernorm_kernel(float* __restrict__ X, const __half* __restrict__ delta,
                                                             const float* __restrict__ w, const float* __restrict__ b,
                                                             __half* __restrict__ out, long long rows) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    constexpr int V = DIM / 128;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    float* xr = X + row * DIM;
    float v[V][4];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int c = k * 128 + lane * 4;
        const float4 t = *reinterpret_cast<const float4*>(xr + c);
        v[k][0] = t.x; v[k][1] = t.y; v[k][2] = t.z; v[k][3] = t.w;
        if (delta) {
            const uint2 raw = *reinterpret_cast<const uint2*>(delta + row * DIM + c);
            const __half2* h = reinterpret_cast<const __half2*>(&raw);
            const float2 d0 = __half22float2(h[0]), d1 = __half22float2(h[1]);
            v[k][0] += d0.x; v[k][1] += d0.y; v[k][2] += d1.x; v[k][3] += d1.y;
            *reinterpret_cast<float4*>(xr + c) = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
        }
        sum += (v[k][0] + v[k][1]) + (v[k][2] + v[k][3]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * (1.f / DIM);
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < V; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float d = v[k][j] - mean;
            sq += d * d;
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq * (1.f / DIM) + 1e-6f);
    if (!out) return;
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int c = k * 128 + lane * 4;
        const float4 wv = __ldg(reinterpret_cast<const float4*>(w + c)), bv = __ldg(reinterpret_cast<const float4*>(b + c));
        __align__(8) __half2 o[2];
        o[0] = __floats2half2_rn((v[k][0] - mean) * rstd * wv.x + bv.x, (v[k][1] - mean) * rstd * wv.y + bv.y);
        o[1] = __floats2half2_rn((v[k][2] - mean) * rstd * wv.z + bv.z, (v[k][3] - mean) * rstd * wv.w + bv.w);
        *reinterpret_cast<uint2*>(out + row * DIM + c) = *reinterpret_cast<const uint2*>(o);
    }
}

// ------------------------------------------------------------------------------------------ flash attention, d = 64
// CTA = 4 warps = 64 query rows of one (image, head); keys/values streamed in blocks of 64 through a 2-stage cp.async
// ring; S and O live in mma.sync accumulator fragments, softmax is online in base 2 (scale*log2e folded into S).
constexpr int FA_D = 64, FA_BM = 64, FA_BN = 64, FA_LD = FA_D + 8;   // +8 halves: conflict-free fragment loads

// BIAS: an additive score bias [heads][N][ldb] fp32, pre-multiplied by log2(e) (BEiT relative position bias, zoe_model.inl);
// ldb >= cdiv(N, 64) * 64 so that the tail block's loads stay in bounds (those columns are masked below)
template <bool BIAS>
__global__ void __launch_bounds__(128) flash_attention_kernel(const __half* __restrict__ qkv, __half* __restrict__ out, int N, int heads,
                                                              const float* __restrict__ bias, int ldb) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    extern __shared__ __align__(16) unsigned char fa_smem[];
    __half* sq = reinterpret_cast<__half*>(fa_smem);            // [64][72]  (later: the output tile)
    __half* sk = sq + FA_BM * FA_LD;                            // [2][64][72]
    __half* sv = sk + 2 * FA_BN * FA_LD;                        // [2][64][72]
    const int dim = heads * FA_D, ld = 3 * dim;
    const int q0 = blockIdx.x * FA_BM, head = blockIdx.y, b = blockIdx.z;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
    const __half* base = qkv + (size_t)b * N * ld + head * FA_D;

    // stage Q (rows clamped; rows >= N are never stored) and the first K/V block
    const int vv = tid & 7, rr = tid >> 3;   // 16-byte column 0..7, row group 0..15
    auto load_kv = [&](int blk, int stage) {
        for (int r = rr; r < FA_BN; r += 16) {
            const int key = min(blk * FA_BN + r, N - 1);
            const __half* src = base + (size_t)key * ld + vv * 8;
            cp_async16(sk + (stage * FA_BN + r) * FA_LD + vv * 8, src + dim);
            cp_async16(sv + (stage * FA_BN + r) * FA_LD + vv * 8, src + 2 * dim);
        }
    };
    for (int r = rr; r < FA_BM; r += 16) cp_async16(sq + r * FA_LD + vv * 8, base + (size_t)min(q0 + r, N - 1) * ld + vv * 8);
    load_kv(0, 0);
    asm volatile("cp.async.commit_group;" ::: "memory");

    const int nblk = (N + FA_BN - 1) / FA_BN;
    const float sl2 = 0.125f * 1.4426950408889634f;   // head_dim**-0.5 * log2(e)
    uint32_t qa[4][4];
    float o[8][4], m[2] = {-1e30f, -1e30f}, l[2] = {0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int r = 0; r < 4; ++r) o[nt][r] = 0.f;

    for (int blk = 0; blk < nblk; ++blk) {
        const int st = blk & 1;
        if (blk + 1 < nblk) load_kv(blk + 1, st ^ 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        if (blk == 0) {
#pragma unroll
            for (int kt = 0; kt < 4; ++kt) {
                const __half* p0 = sq + (warp * 16 + g) * FA_LD + kt * 16 + 2 * t4;
                qa[kt][0] = *reinterpret_cast<const uint32_t*>(p0);
                qa[kt][1] = *reinterpret_cast<const uint32_t*>(p0 + 8 * FA_LD);
                qa[kt][2] = *reinterpret_cast<const uint32_t*>(p0 + 8);
                qa[kt][3] = *reinterpret_cast<const uint32_t*>(p0 + 8 * FA_LD + 8);
            }
        }
        const __half* kb = sk + st * FA_BN * FA_LD;
        const __half* vb = sv + st * FA_BN * FA_LD;
        float s[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
            for (int kt = 0; kt < 4; ++kt) {
                const __half* pk = kb + (nt * 8 + g) * FA_LD + kt * 16 + 2 * t4;
                mma16816(s[nt], qa[kt], *reinterpret_cast<const uint32_t*>(pk), *reinterpret_cast<const uint32_t*>(pk + 8));
            }
        }
        const bool tail = (blk + 1) * FA_BN > N;
        float mx[2] = {m[0], m[1]};
        if (BIAS) {
            // thread's rows q0 + warp*16 + g (+8) (clamped: rows >= N are never stored), columns blk*64 + nt*8 + 2*t4 (+1)
            const float* b0 = bias + ((size_t)head * N + min(q0 + warp * 16 + g, N - 1)) * ldb + blk * FA_BN + 2 * t4;
            const float* b1 = bias + ((size_t)head * N + min(q0 + warp * 16 + g + 8, N - 1)) * ldb + blk * FA_BN + 2 * t4;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float2 u0 = __ldg(reinterpret_cast<const float2*>(b0 + nt * 8));
                const float2 u1 = __ldg(reinterpret_cast<const float2*>(b1 + nt * 8));
                s[nt][0] = fmaf(s[nt][0], sl2, u0.x); s[nt][1] = fmaf(s[nt][1], sl2, u0.y);
                s[nt][2] = fmaf(s[nt][2], sl2, u1.x); s[nt][3] = fmaf(s[nt][3], sl2, u1.y);
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float v = BIAS ? s[nt][r] : s[nt][r] * sl2;
                if (tail && blk * FA_BN + nt * 8 + 2 * t4 + (r & 1) >= N) v = -1e30f;
                s[nt][r] = v;
                mx[r >> 1] = fmaxf(mx[r >> 1], v);
            }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 1));
            mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 2));
        }
        const float a0 = ex2(m[0] - mx[0]), a1 = ex2(m[1] - mx[1]);
        m[0] = mx[0]; m[1] = mx[1];
        float ps[2] = {0.f, 0.f};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float p = ex2(s[nt][r] - mx[r >> 1]);
                s[nt][r] = p;
                ps[r >> 1] += p;
            }
        l[0] = l[0] * a0 + ps[0];
        l[1] = l[1] * a1 + ps[1];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) { o[nt][0] *= a0; o[nt][1] *= a0; o[nt][2] *= a1; o[nt][3] *= a1; }
        // O += P V  (P as fp16 A fragments straight from the accumulators)
#pragma unroll
        for (int kt = 0; kt < 4; ++kt) {
            uint32_t a[4];
            a[0] = pack_half2(s[2 * kt][0], s[2 * kt][1]);
            a[1] = pack_half2(s[2 * kt][2], s[2 * kt][3]);
            a[2] = pack_half2(s[2 * kt + 1][0], s[2 * kt + 1][1]);
            a[3] = pack_half2(s[2 * kt + 1][2], s[2 * kt + 1][3]);
            const __half* pv = vb + (kt * 16 + (lane & 15)) * FA_LD;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                uint32_t b0, b1;
                ldmatrix_x2_trans(b0, b1, pv + nt * 8);
                mma16816(o[nt], a, b0, b1);
            }
        }
        __syncthreads();   // everyone is done with stage `st` before the next iteration's prefetch overwrites it
    }
    // row sums across the quad, normalise, stage through sq (Q is dead), 16-byte stores
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        l[h] += __shfl_xor_sync(0xffffffffu, l[h], 1);
        l[h] += __shfl_xor_sync(0xffffffffu, l[h], 2);
    }
    const float i0 = 1.f / l[0], i1 = 1.f / l[1];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<uint32_t*>(sq + (warp * 16 + g) * FA_LD + nt * 8 + 2 * t4) = pack_half2(o[nt][0] * i0, o[nt][1] * i0);
        *reinterpret_cast<uint32_t*>(sq + (warp * 16 + g + 8) * FA_LD + nt * 8 + 2 * t4) = pack_half2(o[nt][2] * i1, o[nt][3] * i1);
    }
    __syncthreads();
    __half* ob = out + (size_t)b * N * dim + head * FA_D;
    for (int r = rr; r < FA_BM; r += 16)
        if (q0 + r < N) *reinterpret_cast<uint4*>(ob + (size_t)(q0 + r) * dim + vv * 8) = *reinterpret_cast<const uint4*>(sq + r * FA_LD + vv * 8);
}

// ------------------------------------------------------------------------------------------ DPT head helpers
__global__ void __launch_bounds__(256) relu_add_kernel(const uint4* __restrict__ x, const uint4* __restrict__ x0, uint4* __restrict__ y,
                                                        uint4* __restrict__ s, long long n8) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n8) return;
    const uint4 a = x[i];
    const __half2* ah = reinterpret_cast<const __half2*>(&a);
    __align__(16) __half2 r[4];
    const __half2 z = __float2half2_rn(0.f);
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] = __hmax2(ah[k], z);
    y[i] = *reinterpret_cast<const uint4*>(r);
    if (s) {
        const uint4 c = x0[i];
        const __half2* ch = reinterpret_cast<const __half2*>(&c);
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // fp16 + fp16 -> fp16 like the reference's autocast tensors
            const float2 fa = __half22float2(ah[k]), fc = __half22float2(ch[k]);
            r[k] = __floats2half2_rn(fa.x + fc.x, fa.y + fc.y);
        }
        s[i] = *reinterpret_cast<const uint4*>(r);
    }
}

// ATen upsample_bilinear2d, align_corners=True: src = dst * (in-1)/(out-1); fp32 interpolation, fp16 storage
__global__ void __launch_bounds__(256) upsample_bilinear_kernel(const __half* __restrict__ x, __half* __restrict__ out, int B, int h, int w,
                                                                 int C8, int H, int W, float sy, float sx) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * H * W * C8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c8 = (int)(i % C8);
    long long r = i / C8;
    const int X = (int)(r % W);
    r /= W;
    const int Y = (int)(r % H), b = (int)(r / H);
    const float fy = __fmul_rn(sy, (float)Y), fx = __fmul_rn(sx, (float)X);
    const int y0 = min((int)fy, h - 1), x0 = min((int)fx, w - 1);
    const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const size_t C = (size_t)C8 * 8;
    const __half* p = x + (size_t)b * h * w * C + (size_t)c8 * 8;
    const uint4 v00 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)y0 * w + x0) * C));
    const uint4 v01 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)y0 * w + x1) * C));
    const uint4 v10 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)y1 * w + x0) * C));
    const uint4 v11 = __ldg(reinterpret_cast<const uint4*>(p + ((size_t)y1 * w + x1) * C));
    const __half2 *a = reinterpret_cast<const __half2*>(&v00), *bq = reinterpret_cast<const __half2*>(&v01);
    const __half2 *c = reinterpret_cast<const __half2*>(&v10), *d = reinterpret_cast<const __half2*>(&v11);
    __align__(16) __half2 o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 fa = __half22float2(a[k]), fb = __half22float2(bq[k]), fc = __half22float2(c[k]), fd = __half22float2(d[k]);
        o[k] = __floats2half2_rn(hy * (hx * fa.x + lx * fb.x) + ly * (hx * fc.x + lx * fd.x),
                                 hy * (hx * fa.y + lx * fb.y) + ly * (hx * fc.y + lx * fd.y));
    }
    *reinterpret_cast<uint4*>(out + (size_t)i * 8) = *reinterpret_cast<const uint4*>(o);
}

__global__ void __launch_bounds__(256) depth_to_space4_kernel(const __half* __restrict__ T, __half* __restrict__ out, int B, int h, int w,
                                                               int c, int cpad) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const long long total = (long long)B * 4 * h * 4 * w * cpad;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int co = (int)(i % cpad);
    long long r = i / cpad;
    const int X = (int)(r % (4 * w));
    r /= 4 * w;
    const int Y = (int)(r % (4 * h)), b = (int)(r / (4 * h));
    __half v = __float2half_rn(0.f);
    if (co < c) v = T[(((size_t)b * h + (Y >> 2)) * w + (X >> 2)) * (16 * c) + ((Y & 3) * 4 + (X & 3)) * c + co];
    out[i] = v;
}

__global__ void __launch_bounds__(256) im2col_s2_kernel(const __half* __restrict__ x, __half* __restrict__ A, int B, int h, int w, int C,
                                                         int ho, int wo) {
    if (threadIdx.x == 0) NB_PDL_TRIGGER();
    const int C8 = C / 8;
    const long long total = (long long)B * ho * wo * 9 * C8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c8 = (int)(i % C8);
    long long r = i / C8;
    const int tap = (int)(r % 9);
    r /= 9;
    const int X = (int)(r % wo);
    r /= wo;
    const int Y = (int)(r % ho), b = (int)(r / ho);
    const int sy = 2 * Y + tap / 3 - 1, sx = 2 * X + tap % 3 - 1;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (sy >= 0 && sy < h && sx >= 0 && sx < w) v = __ldg(reinterpret_cast<const uint4*>(x + (((size_t)b * h + sy) * w + sx) * C + c8 * 8));
    *reinterpret_cast<uint4*>(A + (size_t)i * 8) = v;
}

template <int C>
__global__ void __launch_bounds__(256) head_final_kernel(const __half* __restrict__ x, const float* __restrict__ wv, float bias,
                                                          float* __restrict__ depth, long long npix) {
    __shared__ float sw[C];
    if (threadIdx.x < C) sw[threadIdx.x] = wv[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const uint4* p = reinterpret_cast<const uint4*>(x + (size_t)i * C);
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < C / 8; ++k) {
        const uint4 v = __ldg(p + k);
        const __half2* hv = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(hv[j]);
            acc = fmaf(f.x, sw[k * 8 + 2 * j], acc);
            acc = fmaf(f.y, sw[k * 8 + 2 * j + 1], acc);
        }
    }
    // the reference's conv output is fp16 under autocast, then ReLU, then .float()
    depth[i] = fmaxf(__half2float(__float2half_rn(acc + bias)), 0.f);
}

// ------------------------------------------------------------------------------------------ host wrappers
int da_patch_im2col(cudaStream_t st, const float* x, int B, int H, int W, __half* A, int kpad) {
    const int ph = H / PATCH, pw = W / PATCH;
    const long long total = (long long)B * ph * pw * kpad;
    patch_im2col_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(x, A, B, H, W, ph, pw, kpad);
    NB_LAUNCHED();
    return 0;
}

int da_assemble_tokens(cudaStream_t st, const __half* T, const float* cls, const float* pos, float* X32, int B, int P, int dim) {
    const long long total = (long long)B * (P + 1) * dim;
    assemble_tokens_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(T, cls, pos, X32, B, P, dim);
    NB_LAUNCHED();
    return 0;
}

int da_add_layernorm(cudaStream_t st, float* X32, const __half* delta, const float* w, const float* b, __half* out, long long rows,
                     int dim) {
    const unsigned grid = (unsigned)cdiv64(rows, 8);
    switch (dim) {
        case 256: add_layernorm_kernel<256><<<grid, 256, 0, st>>>(X32, delta, w, b, out, rows); break;
        case 384: add_layernorm_kernel<384><<<grid, 256, 0, st>>>(X32, delta, w, b, out, rows); break;
        case 768: add_layernorm_kernel<768><<<grid, 256, 0, st>>>(X32, delta, w, b, out, rows); break;
        case 1024: add_layernorm_kernel<1024><<<grid, 256, 0, st>>>(X32, delta, w, b, out, rows); break;
        default: return fail("da_add_layernorm: unsupported embedding dim");
    }
    NB_LAUNCHED();
    return 0;
}

int da_attention(cudaStream_t st, const __half* qkv, __half* out, int B, int N, int heads, const float* bias_log2e, int ldb) {
    const size_t smem = (size_t)(FA_BM + 4 * FA_BN) * FA_LD * sizeof(__half);
    const double T = (double)B * N * heads * FA_D;
    ProfScope ps(st, PC_ATTN, 4.0 * T * N, T * 3 * 2 + (bias_log2e ? (double)heads * N * N * 4 : 0.0), T * 2);
    if (bias_log2e) {
        NB_CHECK(ldb % 2 == 0 && ldb >= cdiv(N, FA_BN) * FA_BN, "bias row stride must be even and cover whole 64-key blocks");
        if (ensure_dyn_smem((const void*)flash_attention_kernel<true>, smem)) return 1;
        flash_attention_kernel<true><<<dim3(cdiv(N, FA_BM), heads, B), 128, smem, st>>>(qkv, out, N, heads, bias_log2e, ldb);
    } else {
        if (ensure_dyn_smem((const void*)flash_attention_kernel<false>, smem)) return 1;
        flash_attention_kernel<false><<<dim3(cdiv(N, FA_BM), heads, B), 128, smem, st>>>(qkv, out, N, heads, nullptr, 0);
    }
    NB_LAUNCHED();
    return 0;
}

int da_relu_add(cudaStream_t st, const __half* x, const __half* x0, __half* y, __half* s, long long n) {
    NB_CHECK(n % 8 == 0, "element count must be a multiple of 8");
    relu_add_kernel<<<(unsigned)cdiv64(n / 8, 256), 256, 0, st>>>(reinterpret_cast<const uint4*>(x), reinterpret_cast<const uint4*>(x0),
                                                                  reinterpret_cast<uint4*>(y), reinterpret_cast<uint4*>(s), n / 8);
    NB_LAUNCHED();
    return 0;
}

int da_upsample_bilinear(cudaStream_t st, const __half* x, int B, int h, int w, int C, __half* out, int H, int W) {
    NB_CHECK(C % 8 == 0, "channels must be a multiple of 8");
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f, sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    const long long total = (long long)B * H * W * (C / 8);
    upsample_bilinear_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(x, out, B, h, w, C / 8, H, W, sy, sx);
    NB_LAUNCHED();
    return 0;
}

int da_depth_to_space4(cudaStream_t st, const __half* T, int B, int h, int w, int c, __half* out, int cpad) {
    const long long total = (long long)B * 16 * h * w * cpad;
    depth_to_space4_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(T, out, B, h, w, c, cpad);
    NB_LAUNCHED();
    return 0;
}

int da_im2col_s2(cudaStream_t st, const __half* x, int B, int h, int w, int C, __half* A) {
    NB_CHECK(C % 8 == 0, "channels must be a multiple of 8");
    const int ho = (h + 1) / 2, wo = (w + 1) / 2;   // floor((h + 2 - 3) / 2) + 1
    const long long total = (long long)B * ho * wo * 9 * (C / 8);
    im2col_s2_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, st>>>(x, A, B, h, w, C, ho, wo);
    NB_LAUNCHED();
    return 0;
}

int da_head_final(cudaStream_t st, const __half* x, long long npix, int C, const float* wv, float bias, float* depth) {
    NB_CHECK(C == 32, "head_final supports 32 input channels");
    head_final_kernel<32><<<(unsigned)cdiv64(npix, 256), 256, 0, st>>>(x, wv, bias, depth, npix);
    NB_LAUNCHED();
    return 0;
}

}  // namespace nb200

using namespace nb200;

// Low-level ops of the depth networks exposed for unit tests (see include/nunif_b200.h).
extern "C" int nb200_vit_attention_f16(const void* qkv, void* out, int B, int N, int heads, const float* bias_log2e, int ldb,
                                       void* stream) {
    NB_CHECK(qkv && out, "null pointer");
    NB_CHECK(B >= 1 && N >= 1 && heads >= 1, "empty attention");
    return da_attention((cudaStream_t)stream, (const __half*)qkv, (__half*)out, B, N, heads, bias_log2e, ldb);
}

extern "C" int nb200_vit_add_layernorm(float* x32, const void* delta, const float* w, const float* b, void* out, long long rows,
                                       int dim, void* stream) {
    NB_CHECK(x32 && (!out || (w && b)), "null pointer");
    NB_CHECK(rows >= 1, "empty input");
    return da_add_layernorm((cudaStream_t)stream, x32, (const __half*)delta, w, b, (__half*)out, rows, dim);
}

extern "C" int nb200_dpt_upsample_bilinear_f16(const void* x, int B, int h, int w, int C, void* out, int H, int W, void* stream) {
    NB_CHECK(x && out, "null pointer");
    NB_CHECK(B >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, "empty image");
    return da_upsample_bilinear((cudaStream_t)stream, (const __half*)x, B, h, w, C, (__half*)out, H, W);
}
