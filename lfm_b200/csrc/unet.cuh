// lfm_b200 - non-GEMM kernels of the ADM UNetModel velocity network (reference models/guided_diffusion/unet.py).
// Activations are NHWC: an fp32 "stream" tensor per block output (skip connections, residual adds) and bf16 operand
// tensors feeding the tcgen05 implicit-GEMM convolutions (gemm2.cuh with a 4-D TMA im2col producer).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace lfm {

// Channel-concatenated view of up to two NHWC fp32 tensors (th.cat([h, hs.pop()], dim=1), unet.py:649 - the
// concatenation is never materialised: GroupNorm reads both sources and writes ONE bf16 operand).
struct Src2 {
    const float* a;
    const float* b;  // may be nullptr
    int Ca, Cb;
};

LFM_DEVICE float4 src2_load(const Src2& s, size_t pix, int ch) {
    if (ch < s.Ca) return *reinterpret_cast<const float4*>(s.a + pix * s.Ca + ch);
    return *reinterpret_cast<const float4*>(s.b + pix * s.Cb + (ch - s.Ca));
}

// ------------------------------------------------------------------------------------------------
// GroupNorm32(32, C) statistics (nn.py:17-19; eps 1e-5, biased variance over (C/32) x H x W per sample).
// grid (nchunk, B): each block reduces a pixel range of one sample into 32 x {sum, sumsq} (fp64 bins),
// partial[b][chunk][32][2].  One warp per pixel; lane l owns channels 128 j + 4 l .. + 3 (C % 128 == 0, so a
// float4 never straddles a group).
constexpr int kGnMaxJ = 16;  // C <= 2048
template <int J>  // J = C / 128 float4 slots per lane per pixel
__global__ void __launch_bounds__(256)
gn_stats_kernel(Src2 s, int HW, int nchunk, double* __restrict__ partial) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    extern __shared__ float s_part[];  // [8 warps][J][32 lanes][2]
    constexpr int C = J * 128, cpg = C / 32;
    constexpr int U = J >= 8 ? 1 : (J >= 4 ? 2 : 4);  // pixels in flight per warp: ~8 independent 512 B requests
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunk = blockIdx.x, b = blockIdx.y;
    const int p0 = static_cast<int>(static_cast<long long>(HW) * chunk / nchunk);
    const int p1 = static_cast<int>(static_cast<long long>(HW) * (chunk + 1) / nchunk);
    float sum[J], sq[J];
#pragma unroll
    for (int j = 0; j < J; ++j) sum[j] = sq[j] = 0.f;
    for (int p = p0 + warp; p < p1; p += 8 * U) {
        float4 v[U][J];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int pp = p + 8 * u;
            const size_t pix = static_cast<size_t>(b) * HW + (pp < p1 ? pp : p);
#pragma unroll
            for (int j = 0; j < J; ++j) v[u][j] = src2_load(s, pix, 128 * j + 4 * lane);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (p + 8 * u < p1) {
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    sum[j] += (v[u][j].x + v[u][j].y) + (v[u][j].z + v[u][j].w);
                    sq[j] += (v[u][j].x * v[u][j].x + v[u][j].y * v[u][j].y) + (v[u][j].z * v[u][j].z + v[u][j].w * v[u][j].w);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < J; ++j) reinterpret_cast<float2*>(s_part)[(warp * J + j) * 32 + lane] = make_float2(sum[j], sq[j]);
    __syncthreads();
    // fixed-order reduction: thread g owns group g = float4 slots [g*cpg/4, (g+1)*cpg/4) of every warp
    if (threadIdx.x < 32) {
        const int g = threadIdx.x;
        const int q0 = g * (cpg / 4), q1 = q0 + cpg / 4;
        double S = 0.0, Q = 0.0;
        for (int w = 0; w < 8; ++w)
            for (int q = q0; q < q1; ++q) {
                const float2 t = reinterpret_cast<const float2*>(s_part)[(w * J + (q >> 5)) * 32 + (q & 31)];
                S += static_cast<double>(t.x);
                Q += static_cast<double>(t.y);
            }
        double* dst = partial + (static_cast<size_t>(b) * nchunk + chunk) * 64 + 2 * g;
        dst[0] = S;
        dst[1] = Q;
    }
}

// GroupNorm apply (+ optional FiLM h*(1+scale)+shift, unet.py:230-234; + optional SiLU) -> bf16 operand.
// Also (optionally) copies the fp32 input through (pre-initialises the ResBlock output for the identity skip,
// unet.py:238 `skip_connection(x) + h`) and/or writes a raw bf16 cast (operand of the 1x1 skip convolution).
struct GnApplyArgs {
    Src2 src;
    const __nv_bfloat16* src_bf16;  // nullptr, or the source as bf16 [B, HW, C] (conv1's output when its fp32 statistics were
                                    // taken in that conv's epilogue: half the bytes to write and to read back)
    int HW, C, nchunk;
    float bins_unit;                 // 1 / the fixed-point scale the producer of `bins` used (GemmEpi::gn_scale): 2^-28 or 2^-22
    const double* partial;
    const unsigned long long* bins;  // nullptr, or fixed-point {sum, sumsq} per (sample, group) from the producing conv
    const float* gamma;
    const float* beta;
    const float* film;  // nullptr, or per-sample [scale(C) | shift(C)] at film + b * film_stride
    int film_stride;
    int act;            // 0 none, 1 SiLU
    float eps;          // 1e-5 (nn.GroupNorm default: ADM / EDM), 1e-6 (VAE decoder)
    __nv_bfloat16* out;
    float* copy_out;            // nullptr or fp32 [B, HW, C]
    __nv_bfloat16* raw_out;     // nullptr or bf16 [B, HW, C]
};
// Per-channel coefficients of one sample: y = x * A[c] + Bc[c] (GroupNorm affine and FiLM folded), into s_coef[2][C].
template <int C>
LFM_DEVICE void gn_coefficients(const GnApplyArgs& a, int b, float* s_coef, float* s_mean, float* s_rstd) {
    constexpr int cpg = C / 32;
    if (threadIdx.x < 32) {
        double S = 0.0, Q = 0.0;
        if (a.bins != nullptr) {  // statistics accumulated by the producing convolution's epilogue (integer, order-free)
            long long si = 0, qi = 0;  // the replicas are integers: their sum is exact whatever the arrival order was
            for (int r = 0; r < kGnBinReplicas; ++r) {
                const unsigned long long* bp = a.bins + (static_cast<size_t>(b) * kGnBinReplicas + r) * 64 + 2 * threadIdx.x;
                si += static_cast<long long>(bp[0]);
                qi += static_cast<long long>(bp[1]);
            }
            S = static_cast<double>(si) * static_cast<double>(a.bins_unit);  // a power of two: exact
            Q = static_cast<double>(qi) * static_cast<double>(a.bins_unit);
        } else {
            for (int c = 0; c < a.nchunk; ++c) {  // fixed order => deterministic
                S += a.partial[(static_cast<size_t>(b) * a.nchunk + c) * 64 + 2 * threadIdx.x];
                Q += a.partial[(static_cast<size_t>(b) * a.nchunk + c) * 64 + 2 * threadIdx.x + 1];
            }
        }
        const double n = static_cast<double>(a.HW) * cpg;
        const double mean = S / n;
        double var = Q / n - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mean[threadIdx.x] = static_cast<float>(mean);
        s_rstd[threadIdx.x] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(a.eps)));
    }
    __syncthreads();
    const float* film = a.film != nullptr ? a.film + static_cast<size_t>(b) * a.film_stride : nullptr;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g = c / cpg;
        float A = s_rstd[g] * a.gamma[c];
        float Bc = a.beta[c] - s_mean[g] * A;
        if (film != nullptr) {  // h * (1 + scale) + shift
            const float sc = 1.f + film[c], sh = film[C + c];
            A *= sc;
            Bc = fmaf(Bc, sc, sh);
        }
        s_coef[c] = A;
        s_coef[C + c] = Bc;
    }
    __syncthreads();
}

// pixels a warp takes per iteration: eight 16-byte loads per lane are issued before the first store (one pixel of C <= 256
// channels is only 1-2 loads per lane: a warp with a single 512-byte request in flight leaves the kernel latency-bound at
// ~40 % of the HBM rate).  Wide channel counts only occur on the small grids; 4 loads keep them inside 64 registers.
__host__ __device__ constexpr int gn_apply_loads(int J) { return J <= 4 ? 8 : 4; }
__host__ __device__ constexpr int gn_apply_pixels(int J) { return J >= gn_apply_loads(J) ? 1 : gn_apply_loads(J) / J; }
template <int J>
__global__ void __launch_bounds__(256, 4)  // 4 blocks per SM resident: the host sizes the grid to ONE wave of 4 x SMs blocks
gn_apply_kernel(GnApplyArgs a) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    extern __shared__ float s_coef[];  // [2][C]
    __shared__ float s_mean[32], s_rstd[32];
    constexpr int C = J * 128;
    constexpr int NL = gn_apply_loads(J);
    constexpr int JB = J >= NL ? NL : J;
    constexpr int PIXB = gn_apply_pixels(J);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.y;
    gn_coefficients<C>(a, b, s_coef, s_mean, s_rstd);
    const bool act = a.act != 0;
    for (int p0 = (blockIdx.x * 8 + warp) * PIXB; p0 < a.HW; p0 += gridDim.x * 8 * PIXB) {
        const size_t pix0 = static_cast<size_t>(b) * a.HW + p0;
#pragma unroll
        for (int j0 = 0; j0 < J; j0 += JB) {
            float4 vv[PIXB][JB];
#pragma unroll
            for (int q = 0; q < PIXB; ++q)
#pragma unroll
                for (int u = 0; u < JB; ++u)
                    if (j0 + u < J && p0 + q < a.HW) {
                        if (a.src_bf16 != nullptr) {
                            const uint2 r = *reinterpret_cast<const uint2*>(a.src_bf16 + (pix0 + q) * C + 128 * (j0 + u) + 4 * lane);
                            const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.x));
                            const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.y));
                            vv[q][u] = make_float4(lo.x, lo.y, hi.x, hi.y);
                        } else {
                            vv[q][u] = src2_load(a.src, pix0 + q, 128 * (j0 + u) + 4 * lane);
                        }
                    }
#pragma unroll
            for (int u = 0; u < JB; ++u) {
                if (j0 + u < J) {
                    const int ch = 128 * (j0 + u) + 4 * lane;
                    const float4 A = *reinterpret_cast<const float4*>(s_coef + ch);
                    const float4 Bc = *reinterpret_cast<const float4*>(s_coef + C + ch);
#pragma unroll
                    for (int q = 0; q < PIXB; ++q) {
                        if (p0 + q < a.HW) {
                            const float4 v = vv[q][u];
                            const size_t off = (pix0 + q) * C + ch;
                            float y0 = fmaf(v.x, A.x, Bc.x), y1 = fmaf(v.y, A.y, Bc.y), y2 = fmaf(v.z, A.z, Bc.z), y3 = fmaf(v.w, A.w, Bc.w);
                            if (act) {
                                y0 = silu_fast(y0), y1 = silu_fast(y1), y2 = silu_fast(y2), y3 = silu_fast(y3);
                            }
                            *reinterpret_cast<uint2*>(a.out + off) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
                            if (a.copy_out != nullptr) *reinterpret_cast<float4*>(a.copy_out + off) = v;
                            if (a.raw_out != nullptr)
                                *reinterpret_cast<uint2*>(a.raw_out + off) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
                        }
                    }
                }
            }
        }
    }
}

// The same pass for a bf16 SOURCE of C <= 512 channels (conv1's output H1; no pass-through copies): 8-byte loads per lane kept
// only half the bytes in flight and ran at 3.6 TB/s where the fp32-source pass reaches 5.5.  Here a warp takes a GROUP of PIXB
// consecutive pixels as one contiguous run of 16-byte chunks (8 channels each; chunk t of the group belongs to lane t % 32), eight
// (six for C = 384) chunks per lane in flight.  HW % PIXB == 0 (checked by the host).
__host__ __device__ constexpr int gn_apply_bf16_pixels(int J) { return J == 1 ? 16 : J == 2 ? 8 : 4; }
template <int J>
__global__ void __launch_bounds__(256, 4)
gn_apply_bf16_kernel(GnApplyArgs a) {
    static_assert(J >= 1 && J <= 4, "C <= 512");
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    extern __shared__ float s_coef[];  // [2][C]
    __shared__ float s_mean[32], s_rstd[32];
    constexpr int C = J * 128;
    constexpr int PIXB = gn_apply_bf16_pixels(J);
    constexpr int NCH = PIXB * J / 2;  // 16-byte chunks per lane per group: 8, 8, 6, 8
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.y;
    gn_coefficients<C>(a, b, s_coef, s_mean, s_rstd);
    const bool act = a.act != 0;
    for (int p0 = (blockIdx.x * 8 + warp) * PIXB; p0 < a.HW; p0 += gridDim.x * 8 * PIXB) {
        const size_t base = (static_cast<size_t>(b) * a.HW + p0) * C;
        uint4 raw[NCH];
#pragma unroll
        for (int i = 0; i < NCH; ++i) raw[i] = *reinterpret_cast<const uint4*>(a.src_bf16 + base + (i * 32 + lane) * 8);
        // chunk i of a lane covers channels (256 i + 8 lane) % C: NSETS different coefficient vectors per lane; take the chunks set
        // by set so that only ONE set (16 registers) is live (the compiler otherwise hoists every set above the loop and spills)
        constexpr int NSETS = J == 4 ? 2 : J == 3 ? 3 : 1;
#pragma unroll
        for (int set = 0; set < NSETS; ++set) {
            if (set > 0) asm volatile("" ::: "memory");
            const int ch = (set * 256 + lane * 8) % C;
            const float4 A0 = *reinterpret_cast<const float4*>(s_coef + ch), A1 = *reinterpret_cast<const float4*>(s_coef + ch + 4);
            const float4 B0 = *reinterpret_cast<const float4*>(s_coef + C + ch), B1 = *reinterpret_cast<const float4*>(s_coef + C + ch + 4);
#pragma unroll
            for (int i = set; i < NCH; i += NSETS) {
                const int e = (i * 32 + lane) * 8;  // element offset inside the group
                const float2 v0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw[i].x));
                const float2 v1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw[i].y));
                const float2 v2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw[i].z));
                const float2 v3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw[i].w));
                float y0 = fmaf(v0.x, A0.x, B0.x), y1 = fmaf(v0.y, A0.y, B0.y), y2 = fmaf(v1.x, A0.z, B0.z), y3 = fmaf(v1.y, A0.w, B0.w);
                float y4 = fmaf(v2.x, A1.x, B1.x), y5 = fmaf(v2.y, A1.y, B1.y), y6 = fmaf(v3.x, A1.z, B1.z), y7 = fmaf(v3.y, A1.w, B1.w);
                if (act) {
                    y0 = silu_fast(y0), y1 = silu_fast(y1), y2 = silu_fast(y2), y3 = silu_fast(y3);
                    y4 = silu_fast(y4), y5 = silu_fast(y5), y6 = silu_fast(y6), y7 = silu_fast(y7);
                }
                *reinterpret_cast<uint4*>(a.out + base + e) =
                    make_uint4(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3), pack_bf16x2(y4, y5), pack_bf16x2(y6, y7));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// input_blocks.0: conv3x3(in_channels=4 -> C), pad 1, NCHW fp32 latents -> NHWC fp32 stream (unet.py:464).
// Network row b reads sample b % x_rows.  One block per output row (b, h); thread = output channel.
__global__ void __launch_bounds__(256)
conv_in_kernel(const float* __restrict__ x, int x_rows, const float* __restrict__ Wt /*[C,4,3,3]*/,
               const float* __restrict__ bias, float* __restrict__ out, int H, int W, int C) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    extern __shared__ float s_in[];  // [4][3][W + 2]
    const int b = blockIdx.x / H, h = blockIdx.x % H;
    const int bs = b % x_rows;
    const int WP = W + 2;
    for (int i = threadIdx.x; i < 4 * 3 * WP; i += blockDim.x) {
        const int c = i / (3 * WP), r = (i / WP) % 3, w = i % WP - 1;
        const int hh = h + r - 1;
        float v = 0.f;
        if (hh >= 0 && hh < H && w >= 0 && w < W) v = x[((static_cast<size_t>(bs) * 4 + c) * H + hh) * W + w];
        s_in[i] = v;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float wreg[36];
#pragma unroll
        for (int i = 0; i < 36; ++i) wreg[i] = __ldg(Wt + static_cast<size_t>(c) * 36 + i);
        const float bc = bias[c];
        for (int w = 0; w < W; ++w) {
            float acc = bc;
#pragma unroll
            for (int ci = 0; ci < 4; ++ci)
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int s = 0; s < 3; ++s) acc = fmaf(wreg[ci * 9 + r * 3 + s], s_in[(ci * 3 + r) * WP + w + s], acc);
            out[((static_cast<size_t>(b) * H + h) * W + w) * C + c] = acc;
        }
    }
}

// Same convolution, register-blocked: a thread owns channel c and walks the output row in strips of 8 pixels; per
// (input channel, filter row) it fetches the 10 input values of the strip with three vector loads (warp-wide
// broadcasts from shared memory) and issues 24 FMAs - 27 instructions per 8 outputs and tap row instead of 48.
// Requires W % 8 == 0 (rows padded to W + 4 floats so that every strip starts 16-byte aligned).
__global__ void __launch_bounds__(256)
conv_in_strip_kernel(const float* __restrict__ x, int x_rows, const float* __restrict__ Wt /*[C,4,3,3]*/,
                     const float* __restrict__ bias, float* __restrict__ out, int H, int W, int C) {
    pdl_wait();
    pdl_trigger();
    extern __shared__ __align__(16) float s_in2[];  // [4][3][W + 4]: position p holds column p - 1
    const int b = blockIdx.x / H, h = blockIdx.x % H;
    const int bs = b % x_rows;
    const int WP = W + 4;
    for (int i = threadIdx.x; i < 4 * 3 * WP; i += blockDim.x) {
        const int c = i / (3 * WP), r = (i / WP) % 3, w = i % WP - 1;
        const int hh = h + r - 1;
        float v = 0.f;
        if (hh >= 0 && hh < H && w >= 0 && w < W) v = x[((static_cast<size_t>(bs) * 4 + c) * H + hh) * W + w];
        s_in2[i] = v;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float wreg[36];
#pragma unroll
        for (int i = 0; i < 36; ++i) wreg[i] = __ldg(Wt + static_cast<size_t>(c) * 36 + i);
        const float bc = bias[c];
        float* orow = out + (static_cast<size_t>(b) * H + h) * W * C + c;
        for (int w0 = 0; w0 < W; w0 += 8) {
            float acc[8];
#pragma unroll
            for (int p = 0; p < 8; ++p) acc[p] = bc;
#pragma unroll
            for (int cr = 0; cr < 12; ++cr) {  // (input channel, filter row)
                const float* ip = s_in2 + cr * WP + w0;
                const float4 a0 = *reinterpret_cast<const float4*>(ip);
                const float4 a1 = *reinterpret_cast<const float4*>(ip + 4);
                const float2 a2 = *reinterpret_cast<const float2*>(ip + 8);
                const float in[10] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y};
                const float k0 = wreg[cr * 3], k1 = wreg[cr * 3 + 1], k2 = wreg[cr * 3 + 2];
#pragma unroll
                for (int p = 0; p < 8; ++p) acc[p] = fmaf(k2, in[p + 2], fmaf(k1, in[p + 1], fmaf(k0, in[p], acc[p])));
            }
#pragma unroll
            for (int p = 0; p < 8; ++p) orow[static_cast<size_t>(w0 + p) * C] = acc[p];
        }
    }
}

// out.2: conv3x3(C -> 4), pad 1, on the GN+SiLU'd bf16 NHWC operand -> NCHW fp32 velocity (unet.py:591-595).
// One warp per output pixel, lane = 8-channel slice; weights [4][9][C] fp32 in shared memory.
__global__ void __launch_bounds__(256)
conv_out_kernel(const __nv_bfloat16* __restrict__ a, const float* __restrict__ Wr /*[4][9][C]*/,
                const float* __restrict__ bias, float* __restrict__ v_out, int B, int H, int W, int C) {
    extern __shared__ float s_w[];
    for (int i = threadIdx.x; i < 36 * C; i += blockDim.x) s_w[i] = Wr[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = B * H * W;
    for (int pix = blockIdx.x * 8 + warp; pix < total; pix += gridDim.x * 8) {
        const int b = pix / (H * W), h = (pix / W) % H, w = pix % W;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int tap = 0; tap < 9; ++tap) {
            const int hh = h + tap / 3 - 1, ww = w + tap % 3 - 1;
            if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;  // warp-uniform
            const __nv_bfloat16* ap = a + (static_cast<size_t>(b) * H * W + static_cast<size_t>(hh) * W + ww) * C;
            for (int c0 = lane * 8; c0 < C; c0 += 256) {
                const uint4 u = *reinterpret_cast<const uint4*>(ap + c0);
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
                float f[8];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 t = __bfloat1622float2(h2[k]);
                    f[2 * k] = t.x, f[2 * k + 1] = t.y;
                }
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    const float* wp = s_w + (o * 9 + tap) * C + c0;
#pragma unroll
                    for (int k = 0; k < 8; ++k) acc[o] = fmaf(f[k], wp[k], acc[o]);
                }
            }
        }
#pragma unroll
        for (int o = 0; o < 4; ++o) acc[o] = warp_sum(acc[o]);
        if (lane < 4) {
            const float r = lane == 0 ? acc[0] : (lane == 1 ? acc[1] : (lane == 2 ? acc[2] : acc[3]));
            v_out[((static_cast<size_t>(b) * 4 + lane) * H + h) * W + w] = r + bias[lane];
        }
    }
}

// out.2 on the tensor cores: the pair GEMM writes [B*H*W, 4] (NHWC); this scatters it to the NCHW velocity.
__global__ void nhwc4_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int HW) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;  // pixel index
    if (i >= static_cast<size_t>(B) * HW) return;
    const float4 v = *reinterpret_cast<const float4*>(in + i * 4);
    const size_t b = i / HW, p = i % HW;
    float* o = out + b * 4 * HW + p;
    o[0] = v.x;
    o[HW] = v.y;
    o[2 * static_cast<size_t>(HW)] = v.z;
    o[3 * static_cast<size_t>(HW)] = v.w;
}

// Upsample: nearest x2 of the fp32 stream -> bf16 operand of the following conv3x3 (unet.py:92-99).
// One thread per INPUT float4: one 16-byte load, four 8-byte stores (the 2 x 2 output pixels); grid (ceil(W * C/4 / 256), B * H),
// so the only index arithmetic is one 32-bit division (the first version decoded a flat 64-bit output index per thread: three
// 64-bit divisions per 8 bytes stored, 2.3 TB/s).
__global__ void __launch_bounds__(256)
upsample2x_cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int H, int W, int C) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const unsigned c4n = static_cast<unsigned>(C) >> 2;
    const unsigned i = blockIdx.x * 256u + threadIdx.x;
    if (i >= static_cast<unsigned>(W) * c4n) return;
    const unsigned w = i / c4n, c4 = i - w * c4n;
    const unsigned bh = blockIdx.y;  // b * H + h
    const unsigned b = bh / static_cast<unsigned>(H), h = bh - b * static_cast<unsigned>(H);
    const float4 v = *reinterpret_cast<const float4*>(x + (static_cast<size_t>(bh) * W + w) * C + c4 * 4);
    const uint2 o = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    __nv_bfloat16* row0 = y + ((static_cast<size_t>(b) * 2 * H + 2 * h) * 2 * W + 2 * w) * C + c4 * 4;
    __nv_bfloat16* row1 = row0 + static_cast<size_t>(2) * W * C;
    *reinterpret_cast<uint2*>(row0) = o;
    *reinterpret_cast<uint2*>(row0 + C) = o;
    *reinterpret_cast<uint2*>(row1) = o;
    *reinterpret_cast<uint2*>(row1 + C) = o;
}

// ------------------------------------------------------------------------------------------------
// AttentionBlock core (QKVAttentionLegacy, unet.py:319-334) for the short token grids of the UNet (T <= 256).
// qkv: bf16 [B*T, 3C] with channel = head*3ch + {q,k,v}*ch + c ; out: bf16 [B*T, C] with channel = head*ch + c.
// One warp per query; lanes split the keys for the scores and the channels for the output.  fp32 softmax.
__global__ void __launch_bounds__(256)
attention_small_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int T, int C, int heads) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    __shared__ float s_q[8][256];
    __shared__ float s_p[8][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x / heads, head = blockIdx.x % heads;
    const int ch = C / heads;
    const int t = blockIdx.y * 8 + warp;
    if (t >= T) return;
    const size_t ld = static_cast<size_t>(3) * C;
    const __nv_bfloat16* base = qkv + static_cast<size_t>(b) * T * ld + static_cast<size_t>(head) * 3 * ch;
    const float scale2 = rsqrtf(static_cast<float>(ch));  // (ch^-1/4)^2
    for (int c = lane; c < ch; c += 32) s_q[warp][c] = __bfloat162float(base[static_cast<size_t>(t) * ld + c]);
    __syncwarp();
    float mx = -INFINITY;
    for (int s = lane; s < T; s += 32) {
        const __nv_bfloat16* kp = base + static_cast<size_t>(s) * ld + ch;
        float acc = 0.f;
        for (int c = 0; c < ch; c += 8) {
            const uint4 u = *reinterpret_cast<const uint4*>(kp + c);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = __bfloat1622float2(h2[k]);
                acc = fmaf(s_q[warp][c + 2 * k], f.x, acc);
                acc = fmaf(s_q[warp][c + 2 * k + 1], f.y, acc);
            }
        }
        acc *= scale2;
        s_p[warp][s] = acc;
        mx = fmaxf(mx, acc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int s = lane; s < T; s += 32) {
        const float p = __expf(s_p[warp][s] - mx);
        s_p[warp][s] = p;
        sum += p;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.f / sum;
    // output channels: lane handles c = 2*lane + 64*m
    for (int c0 = 2 * lane; c0 < ch; c0 += 64) {
        float a0 = 0.f, a1 = 0.f;
        const __nv_bfloat16* vp = base + 2 * ch + c0;
        for (int s = 0; s < T; ++s) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(vp + static_cast<size_t>(s) * ld));
            const float p = s_p[warp][s];
            a0 = fmaf(p, f.x, a0);
            a1 = fmaf(p, f.y, a1);
        }
        *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(b) * T + t) * C + head * ch + c0) = pack_bf16x2(a0 * inv, a1 * inv);
    }
}

// Split-K epilogue: out[m, n] (+)= bias[n] + sum_s partial[s][m][n], slabs added in a fixed order (deterministic).
__global__ void splitk_reduce_kernel(const float* __restrict__ partial, int S, size_t slab /*elements*/, const float* __restrict__ bias,
                                     float* out, int N, size_t n4, int accumulate, const float* addend /* nullable; may alias out */) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias) + (i % (N / 4)));
    float4 acc = b4;
    for (int s = 0; s < S; ++s) {
        const float4 v = *reinterpret_cast<const float4*>(partial + s * slab + i * 4);
        acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
    }
    float4* op = reinterpret_cast<float4*>(out) + i;
    if (addend != nullptr) {
        const float4 a = *(reinterpret_cast<const float4*>(addend) + i);
        acc.x += a.x, acc.y += a.y, acc.z += a.z, acc.w += a.w;
    }
    if (accumulate) {
        const float4 o = *op;
        acc.x += o.x, acc.y += o.y, acc.z += o.z, acc.w += o.w;
    }
    *op = acc;
}

// Same computation with K and V of the (sample, head) staged ONCE in shared memory (rows padded by 16 bytes so the
// 16-byte per-lane key reads are bank-conflict free); 8 warps share them, one query per warp at a time.
// Used when (2 T ch + pad) bf16 fit in shared memory (all LFM presets: T <= 64, ch <= 256).
__global__ void __launch_bounds__(256)
attention_small_smem_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int T, int C, int heads) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    extern __shared__ __align__(16) uint8_t s_kv[];
    __shared__ float s_q[8][256];
    __shared__ float s_p[8][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x / heads, head = blockIdx.x % heads;
    const int ch = C / heads;
    const int rs = ch * 2 + 16;  // padded row stride in bytes
    uint8_t* sK = s_kv;
    uint8_t* sV = s_kv + static_cast<size_t>(T) * rs;
    const size_t ld = static_cast<size_t>(3) * C;
    const __nv_bfloat16* base = qkv + static_cast<size_t>(b) * T * ld + static_cast<size_t>(head) * 3 * ch;
    const int cpr = ch / 8;  // 16-byte chunks per row
    for (int i = threadIdx.x; i < T * cpr; i += 256) {
        const int s = i / cpr, c = (i % cpr) * 8;
        *reinterpret_cast<uint4*>(sK + s * rs + c * 2) = *reinterpret_cast<const uint4*>(base + static_cast<size_t>(s) * ld + ch + c);
        *reinterpret_cast<uint4*>(sV + s * rs + c * 2) = *reinterpret_cast<const uint4*>(base + static_cast<size_t>(s) * ld + 2 * ch + c);
    }
    __syncthreads();
    const float scale2 = rsqrtf(static_cast<float>(ch));
    for (int t = warp; t < T; t += 8) {
        for (int c = lane; c < ch; c += 32) s_q[warp][c] = __bfloat162float(base[static_cast<size_t>(t) * ld + c]);
        __syncwarp();
        float mx = -INFINITY;
        for (int s = lane; s < T; s += 32) {
            const uint8_t* kp = sK + s * rs;
            float acc = 0.f;
            for (int c = 0; c < ch; c += 8) {
                const uint4 u = *reinterpret_cast<const uint4*>(kp + c * 2);
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = __bfloat1622float2(h2[k]);
                    acc = fmaf(s_q[warp][c + 2 * k], f.x, acc);
                    acc = fmaf(s_q[warp][c + 2 * k + 1], f.y, acc);
                }
            }
            acc *= scale2;
            s_p[warp][s] = acc;
            mx = fmaxf(mx, acc);
        }
        mx = warp_max(mx);
        float sum = 0.f;
        for (int s = lane; s < T; s += 32) {
            const float p = __expf(s_p[warp][s] - mx);
            s_p[warp][s] = p;
            sum += p;
        }
        sum = warp_sum(sum);
        __syncwarp();
        const float inv = 1.f / sum;
        for (int c0 = 2 * lane; c0 < ch; c0 += 64) {
            float a0 = 0.f, a1 = 0.f;
            const uint8_t* vp = sV + c0 * 2;
#pragma unroll 4
            for (int s = 0; s < T; ++s) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(vp + s * rs));
                const float p = s_p[warp][s];
                a0 = fmaf(p, f.x, a0);
                a1 = fmaf(p, f.y, a1);
            }
            *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(b) * T + t) * C + head * ch + c0) = pack_bf16x2(a0 * inv, a1 * inv);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// Attention core for the short token grids (T = 16 or 64 tokens per sample) on the tensor cores: warp-level
// mma.sync m16n8k16 (bf16 in, fp32 accumulate) - these tiles are far too small for a tcgen05 pipeline, and the SIMT
// kernels above are instruction-issue bound (about 1000 warp instructions per query).  Same layouts as
// attention_small_kernel: qkv [B*T, 3C] with channel = head*3ch + {q,k,v}*ch + c, out [B*T, C].
// One warp owns 16 query rows: S = Q K^T stays in registers, softmax on the accumulator fragments (fp32), the bf16
// probabilities are re-used directly as the A fragments of P V (no shared-memory round trip).
// T = 64: one (sample, head) per 4-warp block; T = 16: four (sample, head) pairs per block, one warp each.
LFM_DEVICE void cp_async_16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
LFM_DEVICE void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
LFM_DEVICE void ldmatrix_x4(uint32_t* r, const void* smem_ptr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem_ptr)));
}
LFM_DEVICE void ldmatrix_x4_trans(uint32_t* r, const void* smem_ptr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem_ptr)));
}
LFM_DEVICE void mma_bf16_16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int T, int CH>
__global__ void __launch_bounds__(128)
attention_mma_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int C, int heads, int n_items,
                     float scale_log2e /* <= 0: CH^-1/2 * log2(e); > 0: given (DiT-XL: CH = 80 is head_dim 72 padded) */) {
    pdl_wait();
    pdl_trigger();
    constexpr int ITEMS = T == 16 ? 4 : 1;  // (sample, head) pairs per block
    static_assert(T == 16 || T == 64, "one or four 16-row warps per (sample, head)");
    constexpr int LD = CH + 8;              // row pitch in elements: +16 bytes keeps ldmatrix bank-conflict free
    constexpr int CPR = CH / 8;             // 16-byte chunks per row
    extern __shared__ __align__(16) uint8_t att_smem[];
    __nv_bfloat16* sm = reinterpret_cast<__nv_bfloat16*>(att_smem);  // [ITEMS][q,k,v][T][LD]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t ld = static_cast<size_t>(3) * C;
    for (int i = threadIdx.x; i < ITEMS * 3 * T * CPR; i += 128) {
        const int c8 = i % CPR;
        int r = i / CPR;
        const int t = r % T;
        r /= T;
        const int which = r % 3, it = r / 3;
        const int item = blockIdx.x * ITEMS + it;
        __nv_bfloat16* dst = sm + (static_cast<size_t>(it * 3 + which) * T + t) * LD + c8 * 8;
        if (item < n_items) {  // asynchronous copies: all of a thread's 16-byte requests are in flight together
            const int b = item / heads, h = item % heads;
            cp_async_16(dst, qkv + (static_cast<size_t>(b) * T + t) * ld + static_cast<size_t>(h) * 3 * CH + which * CH + c8 * 8);
        } else {
            *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    cp_async_wait_all();
    __syncthreads();
    const int it = ITEMS == 1 ? 0 : warp;
    const int item = blockIdx.x * ITEMS + it;
    if (item >= n_items) return;
    const int r0 = ITEMS == 1 ? warp * 16 : 0;
    const __nv_bfloat16* sQ = sm + static_cast<size_t>(it * 3 + 0) * T * LD;
    const __nv_bfloat16* sK = sm + static_cast<size_t>(it * 3 + 1) * T * LD;
    const __nv_bfloat16* sV = sm + static_cast<size_t>(it * 3 + 2) * T * LD;

    float acc_s[T / 8][4];
#pragma unroll
    for (int j = 0; j < T / 8; ++j) acc_s[j][0] = acc_s[j][1] = acc_s[j][2] = acc_s[j][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < CH / 16; ++kk) {
        uint32_t a[4];
        ldmatrix_x4(a, sQ + (r0 + (lane & 15)) * LD + kk * 16 + (lane >> 4) * 8);
#pragma unroll
        for (int j2 = 0; j2 < T / 16; ++j2) {
            uint32_t bk[4];
            ldmatrix_x4(bk, sK + (j2 * 16 + (lane & 7) + ((lane >> 4) << 3)) * LD + kk * 16 + ((lane >> 3) & 1) * 8);
            mma_bf16_16816(acc_s[2 * j2], a, bk[0], bk[1]);
            mma_bf16_16816(acc_s[2 * j2 + 1], a, bk[2], bk[3]);
        }
    }
    // softmax over the keys of rows g = lane / 4 (values [0], [1]) and g + 8 ([2], [3]); a row lives in one quad
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < T / 8; ++j) {
        m0 = fmaxf(m0, fmaxf(acc_s[j][0], acc_s[j][1]));
        m1 = fmaxf(m1, fmaxf(acc_s[j][2], acc_s[j][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    const float sl2 = scale_log2e > 0.f ? scale_log2e
                                        : rsqrtf(static_cast<float>(CH)) * 1.4426950408889634f;  // (ch^-1/4)^2 = 1/sqrt(ch), in log2 units
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int j = 0; j < T / 8; ++j) {
        acc_s[j][0] = exp2f((acc_s[j][0] - m0) * sl2);
        acc_s[j][1] = exp2f((acc_s[j][1] - m0) * sl2);
        acc_s[j][2] = exp2f((acc_s[j][2] - m1) * sl2);
        acc_s[j][3] = exp2f((acc_s[j][3] - m1) * sl2);
        l0 += acc_s[j][0] + acc_s[j][1];
        l1 += acc_s[j][2] + acc_s[j][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);

    float acc_o[CH / 8][4];
#pragma unroll
    for (int n = 0; n < CH / 8; ++n) acc_o[n][0] = acc_o[n][1] = acc_o[n][2] = acc_o[n][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < T / 16; ++kk) {
        uint32_t pa[4];
        pa[0] = pack_bf16x2(acc_s[2 * kk][0], acc_s[2 * kk][1]);
        pa[1] = pack_bf16x2(acc_s[2 * kk][2], acc_s[2 * kk][3]);
        pa[2] = pack_bf16x2(acc_s[2 * kk + 1][0], acc_s[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(acc_s[2 * kk + 1][2], acc_s[2 * kk + 1][3]);
#pragma unroll
        for (int n2 = 0; n2 < CH / 16; ++n2) {
            uint32_t bv[4];
            ldmatrix_x4_trans(bv, sV + (kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + n2 * 16 + (lane >> 4) * 8);
            mma_bf16_16816(acc_o[2 * n2], pa, bv[0], bv[1]);
            mma_bf16_16816(acc_o[2 * n2 + 1], pa, bv[2], bv[3]);
        }
    }
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    const int b = item / heads, h = item % heads;
    const int row = r0 + (lane >> 2);
    __nv_bfloat16* o0 = out + (static_cast<size_t>(b) * T + row) * C + static_cast<size_t>(h) * CH + (lane & 3) * 2;
    __nv_bfloat16* o1 = o0 + static_cast<size_t>(8) * C;
#pragma unroll
    for (int n = 0; n < CH / 8; ++n) {
        *reinterpret_cast<uint32_t*>(o0 + n * 8) = pack_bf16x2(acc_o[n][0] * inv0, acc_o[n][1] * inv0);
        *reinterpret_cast<uint32_t*>(o1 + n * 8) = pack_bf16x2(acc_o[n][2] * inv1, acc_o[n][3] * inv1);
    }
}

// ------------------------------------------------------------------------------------------------
// EDM-style ADM (DhariwalUNet, reference models/EDM.py) additions.
//
// Resampling inside a UNetBlock (EDM.py:101-134 with resample_filter [1, 1]): `down` = 2x2 mean, `up` = nearest x2.
// One launch moves BOTH tensors of the block to the new resolution: the GroupNorm+SiLU'd bf16 operand of conv0 and
// the fp32 stream that becomes the (weight-free, kernel = 0) skip branch.  Index space = output pixels x C/4.
template <bool UP>
__global__ void resample2x_kernel(const __nv_bfloat16* __restrict__ a_in, __nv_bfloat16* __restrict__ a_out,
                                  const float* __restrict__ x_in, float* __restrict__ x_out, int B, int H, int W, int C) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const int Ho = UP ? 2 * H : H / 2, Wo = UP ? 2 * W : W / 2;
    const size_t n4 = static_cast<size_t>(B) * Ho * Wo * (C / 4);  // < 2^32 (checked by the host): 32-bit index arithmetic
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const unsigned c4n = static_cast<unsigned>(C) >> 2, i32 = static_cast<unsigned>(i);
    unsigned r = i32 / c4n;
    const int c = static_cast<int>(i32 - r * c4n) * 4;
    const unsigned r2 = r / static_cast<unsigned>(Wo);
    const int wo = static_cast<int>(r - r2 * Wo);
    const int b = static_cast<int>(r2 / static_cast<unsigned>(Ho));
    const int ho = static_cast<int>(r2 - static_cast<unsigned>(b) * Ho);
    if (UP) {
        const size_t src = ((static_cast<size_t>(b) * H + ho / 2) * W + wo / 2) * C + c;
        *reinterpret_cast<uint2*>(a_out + i * 4) = *reinterpret_cast<const uint2*>(a_in + src);
        *reinterpret_cast<float4*>(x_out + i * 4) = *reinterpret_cast<const float4*>(x_in + src);
    } else {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), xs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
                const size_t src = ((static_cast<size_t>(b) * H + 2 * ho + dy) * W + 2 * wo + dx) * C + c;
                const uint2 u = *reinterpret_cast<const uint2*>(a_in + src);
                const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
                const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
                acc.x += f0.x, acc.y += f0.y, acc.z += f1.x, acc.w += f1.y;
                const float4 v = *reinterpret_cast<const float4*>(x_in + src);
                xs.x += v.x, xs.y += v.y, xs.z += v.z, xs.w += v.w;
            }
        *reinterpret_cast<uint2*>(a_out + i * 4) =
            make_uint2(pack_bf16x2(0.25f * acc.x, 0.25f * acc.y), pack_bf16x2(0.25f * acc.z, 0.25f * acc.w));
        *reinterpret_cast<float4*>(x_out + i * 4) = make_float4(0.25f * xs.x, 0.25f * xs.y, 0.25f * xs.z, 0.25f * xs.w);
    }
}

// UNetBlock.qkv rows (EDM.py:277-281: out-channel = head*3dh + c*3 + {q,k,v}) re-ordered at load time into the
// layout of the attention kernel that will consume them:
//   mode 0  head*3dh + {q,k,v}*dh + c   (attention_small*_kernel, the guided-diffusion "legacy" order)
//   mode 1  {q,k,v}*C + head*dh + c     (attention3_t256_d64, the DiT order)
LFM_DEVICE int edm_qkv_src_row(int r, int C, int dh, int mode) {
    int h, w, c;
    if (mode == 0) {
        h = r / (3 * dh), w = (r % (3 * dh)) / dh, c = r % dh;
    } else {
        w = r / C, h = (r % C) / dh, c = r % dh;
    }
    return h * 3 * dh + c * 3 + w;
}
__global__ void edm_qkv_weight_repack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int C, int dh, int mode) {
    const size_t n = static_cast<size_t>(3) * C * C;
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = static_cast<int>(i / C), k = static_cast<int>(i % C);
    out[i] = __float2bfloat16(w[static_cast<size_t>(edm_qkv_src_row(r, C, dh, mode)) * C + k]);
}
__global__ void edm_qkv_bias_repack_kernel(const float* __restrict__ b, float* __restrict__ out, int C, int dh, int mode) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= 3 * C) return;
    out[r] = b[edm_qkv_src_row(r, C, dh, mode)];
}

// Labels of one network batch for the one-hot column gather of map_label (EDM.py:822-829): row b reads table row
// y[b]; under forward_with_cfg (drop_half_label) rows >= rows/2 read the all-zero row `null_row`.
__global__ void edm_labels_kernel(const long long* __restrict__ y, long long* __restrict__ out, int rows, int drop_from, int null_row) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= rows) return;
    long long v = y[b];
    if (b >= drop_from || v < 0 || v >= null_row) v = null_row;
    out[b] = v;
}

// conv weight repack: [Cout, Cin, 3, 3] fp32 -> [Cout, 3, 3, Cin] bf16 (K index = (r*3+s)*Cin + c, K-major rows)
__global__ void conv_weight_repack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int Cout, int Cin, int taps) {
    const size_t n = static_cast<size_t>(Cout) * Cin * taps;
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = static_cast<int>(i % Cin);
    const int tap = static_cast<int>((i / Cin) % taps);
    const int o = static_cast<int>(i / (static_cast<size_t>(Cin) * taps));
    out[i] = __float2bfloat16(w[(static_cast<size_t>(o) * Cin + c) * taps + tap]);
}
// out.2 weight repack: [4, C, 3, 3] fp32 -> [4][9][C] fp32
__global__ void conv_out_weight_repack_kernel(const float* __restrict__ w, float* __restrict__ out, int C) {
    const int n = 4 * 9 * C;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = i % C, tap = (i / C) % 9, o = i / (9 * C);
    out[i] = w[(static_cast<size_t>(o) * C + c) * 9 + tap];
}

// sinusoidal timestep features of arbitrary even width (nn.py:103-121; cos first, raw t)
__global__ void timestep_features_dim_kernel(const float* __restrict__ t, int t_numel, float* __restrict__ tf, int B, int dim) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const int b = blockIdx.x;
    const int half = dim / 2;
    for (int i = threadIdx.x; i < dim; i += blockDim.x) {
        const float tv = t[t_numel == 1 ? 0 : b];
        const int k = i < half ? i : i - half;
        const float freq = expf(-9.210340371976184f * static_cast<float>(k) / static_cast<float>(half));
        const float a = tv * freq;
        tf[static_cast<size_t>(b) * dim + i] = (i < half) ? cosf(a) : sinf(a);
    }
}

// general skinny linear (any K % 4 == 0): out[b, j] = act(bias[j] + W[j,:] . in[b,:] (+ table[idx[b], j]))
// mode 0: SiLU -> fp32;  mode 1: (+table) then SiLU -> bf16
__global__ void __launch_bounds__(256)
skinny_linear_gen_kernel(const float* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ in, int B,
                         int N, int K, const float* __restrict__ table, const long long* __restrict__ idx, int mode,
                         float* __restrict__ out_f32, __nv_bfloat16* __restrict__ out_bf16, int max_row) {
    pdl_wait();  // PDL: nothing of the previous kernel's output is touched above this line
    pdl_trigger();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * 8 + warp;
    if (j >= N) return;
    const float4* wp = reinterpret_cast<const float4*>(W + static_cast<size_t>(j) * K);
    const float bj = bias[j];
    for (int b = 0; b < B; ++b) {
        const float4* ip = reinterpret_cast<const float4*>(in + static_cast<size_t>(b) * K);
        float acc = 0.f;
        for (int m = lane; m < K / 4; m += 32) {
            const float4 w4 = __ldg(wp + m), x4 = __ldg(ip + m);
            acc = fmaf(w4.x, x4.x, acc);
            acc = fmaf(w4.y, x4.y, acc);
            acc = fmaf(w4.z, x4.z, acc);
            acc = fmaf(w4.w, x4.w, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) {
            float v = acc + bj;
            if (mode == 1 && table != nullptr && idx != nullptr) {
                long long row = idx[b];
                row = row < 0 ? 0 : (row > max_row ? max_row : row);  // never read outside the table
                v += table[static_cast<size_t>(row) * N + j];
            }
            v = silu(v);
            if (mode == 0)
                out_f32[static_cast<size_t>(b) * N + j] = v;
            else
                out_bf16[static_cast<size_t>(b) * N + j] = __float2bfloat16(v);
        }
    }
}

}  // namespace lfm
