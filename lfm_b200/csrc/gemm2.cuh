// lfm_b200 - 2-CTA (cta_group::2) persistent tcgen05 GEMM: the workhorse for the DiT linear layers.
//
//   C[M, N] = A[M, K] * W[N, K]^T,  one 256 x 256 output tile per CTA PAIR (thread-block cluster of 2).
//
// Why pairs: with one CTA per 128 x 256 tile every SM pulls 48 KB per 64-wide K slab from L2 (94 B/clk/SM at
// full tensor rate) and the measured tensor-pipe utilisation tops out at ~65 % (profiles/r1_gemm_full.md).  In
// cta_group::2 mode each CTA stages only its own 128 rows of A and HALF of the W tile (128 of the 256 rows); the
// tensor cores of both SMs read the two halves from both shared memories.  32 KB per slab per SM (64 B/clk), and
// the freed shared memory deepens the TMA ring from 4 to 6 stages.
//
// Roles per CTA (384 threads): warp 0 = TMA producer (own A rows + own half of W; completion bytes are posted
// on the LEADER CTA's mbarrier), warp 1 = MMA issuer (leader CTA only, tcgen05.mma.cta_group::2, M = 256),
// warp 2 = TMEM allocator, warps 4..11 = epilogue: 8 warps, TMEM lane quadrant = warp % 4, column half =
// (warp - 4) / 4, software-pipelined tcgen05.ld (next chunk in flight while the current one is processed).
// Accumulator double-buffered in TMEM (2 x 256 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include "common.cuh"
#include "gemm.cuh"

namespace lfm {

constexpr int kG2Threads = 384;
constexpr int kG2ThreadsFin = 512;  // + 4 LayerNorm finisher warps (warps 12..15)
constexpr int kG2BlockN = 256;
constexpr int kG2Stages = 6;
constexpr int kG2ABytes = 128 * 64 * 2;
constexpr int kG2BBytes = 128 * 64 * 2;  // this CTA's half of the W tile
constexpr int kG2StageBytes = kG2ABytes + kG2BBytes;
constexpr int kG2StagingBytes = 8 * 4096;  // one 32-row x 128-byte tile per epilogue warp
constexpr int kG2SmemBytes = kG2Stages * kG2StageBytes + 1024 /*barriers*/ + kG2StagingBytes + 1024 /*align slack*/;

LFM_DEVICE uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
LFM_DEVICE void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster
LFM_DEVICE void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// TMA load issued by either CTA of the pair; the transaction bytes are credited to the LEADER CTA's mbarrier
// (shared::cluster address of the executing CTA with the CTA-rank bit cleared).
LFM_DEVICE void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1) {
    const uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar), "r"(c0), "r"(c1)
        : "memory");
}
LFM_DEVICE void tma_load_2d_2sm_hint(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1, uint64_t policy) {
    const uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
// 4-D variant (NHWC activation tensor {C, W, H, B}): the im2col gather of one filter tap is a shifted box;
// out-of-bounds rows/columns (the zero padding) are zero-filled by TMA.
LFM_DEVICE void tma_load_4d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2,
                                int32_t c3) {
    const uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// Implicit-GEMM convolution geometry (taps == 0: plain GEMM, A is a 2-D [M, K] matrix).
// Output pixels are flattened (b, h, w) row-major; a CTA's 128 output rows are whole image rows (W * rows == 128),
// whole images (H * W divides 128) or one 128-pixel segment of an image row (W = 256 or 512, a multiple of 128: the last
// stages of the VAE decoder - 2 or 4 segments per row), so the matching input window of tap (r, s) is ONE 4-D box.
struct ConvGeom {
    int taps;     // 0 (GEMM), 9 (3x3, pad 1)
    int cblocks;  // C_in / 64
    int W;        // OUTPUT width
    int HW;       // OUTPUT height * width
    int stride;   // 1 or 2 (the tensor map carries the matching element strides)
    // Batched GEMM (taps == 0, batch_m > 0): the M rows are batch_m-row groups; group g multiplies against ITS OWN
    // block of W rows, [g * b_batch_rows, g * b_batch_rows + N)  - e.g. S_g = Q_g K_g^T per image.  a_mod > 0: the A
    // operand is shared by all groups (A row = row % a_mod) - e.g. V_g^T = W_v X_g^T.  batch_m % 256 == 0, N % 256 == 0.
    int batch_m = 0;
    int a_mod = 0;
    int b_batch_rows = 0;
};

LFM_DEVICE void umma_ss_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// commit -> arrive on the mbarrier at this offset in BOTH CTAs of the pair
LFM_DEVICE void umma_commit_2cta(uint64_t* bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
template <uint32_t kCols>
LFM_DEVICE void tmem_alloc_2cta(uint32_t* smem_result) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
LFM_DEVICE void tmem_dealloc_2cta(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// TMA reduce-add shared -> global (fp32 tensor map): global[tile] += smem[tile], performed at L2.
LFM_DEVICE void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}

LFM_DEVICE void tma_reduce_add_2d_hint(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1, uint64_t policy) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(policy)
                 : "memory");
}

// Epilogue math for 32 accumulator columns of one row -> f[32] (bias, GELU, gate).
template <int EPI>
LFM_DEVICE void epilogue_math(const uint32_t* v, float* f, const GemmEpi& ep, int n0, int N, const float* gate_row,
                              const float* add_row = nullptr) {
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
    if (n0 >= N) return;  // warp-uniform; the TMA store clips these columns anyway
    if (EPI == EPI_BIAS_F32 && add_row != nullptr) {  // residual connection added here (see GemmEpi::addend)
        const float4* ap = reinterpret_cast<const float4*>(add_row + n0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (n0 + j * 4 < N) {
                const float4 a4 = __ldcg(ap + j);
                f[4 * j + 0] += a4.x;
                f[4 * j + 1] += a4.y;
                f[4 * j + 2] += a4.z;
                f[4 * j + 3] += a4.w;
            }
        }
    }
    if (ep.bias != nullptr) {
        const float4* bp = reinterpret_cast<const float4*>(ep.bias + n0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (n0 + j * 4 < N) {
                const float4 b4 = __ldg(bp + j);
                add_x2(f[4 * j + 0], f[4 * j + 1], b4.x, b4.y);
                add_x2(f[4 * j + 2], f[4 * j + 3], b4.z, b4.w);
            }
        }
    }
    if (EPI == EPI_BIAS_GELU_BF16) {
#pragma unroll
        for (int j = 0; j < 32; j += 2) gelu_tanh_x2(f[j], f[j + 1]);
    }
    if (EPI == EPI_GATE_RESID_F32 && gate_row != nullptr) {
        const float4* gp = reinterpret_cast<const float4*>(gate_row + n0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (n0 + j * 4 < N) {
                const float4 g4 = __ldg(gp + j);
                mul_x2(f[4 * j + 0], f[4 * j + 1], g4.x, g4.y);
                mul_x2(f[4 * j + 2], f[4 * j + 3], g4.z, g4.w);
            }
        }
    }
}

// GroupNorm statistics of one 32-column chunk (see GemmEpi::gn_bins): per-thread sums over each group's columns, then ONE
// halving butterfly over the 32 rows for all V = 2 * groups values at once - at every step a lane keeps half of its values and
// hands the other half to its partner, so 16 values cost 8 + 4 + 2 + 1 + 1 = 16 shuffles (one warp_sum per value: 80) and end up
// on 16 different lanes, which issue their 64-bit integer atomics in ONE instruction.  (The first version - a warp_sum and a
// lane-0 atomic per value - made a 128-channel convolution's epilogue cost more than its mainloop: 866 us vs 406 us.)
template <int V>
LFM_DEVICE float halving_reduce(float (&v)[V], int lane) {
    int width = V;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        if (width > 1) {
            width >>= 1;
            const bool hi = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < V / 2; ++i)
                if (i < width) {
                    const float send = hi ? v[i] : v[i + width];
                    const float keep = hi ? v[i + width] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
        }
    }
    return v[0];  // the total of value (lane >> (5 - log2 V)); every lane of that group of lanes holds it
}
template <int CPG>
LFM_DEVICE void gn_accumulate_chunk(const float* f, bool row_ok, int n0, unsigned long long* bins_b, int lane, double scale) {
    constexpr int NG = CPG >= 32 ? 1 : 32 / CPG;   // groups inside this chunk
    constexpr int W = CPG >= 32 ? 32 : CPG;        // columns per group inside this chunk
    constexpr int V = 2 * NG;                      // {sum, sum of squares} per group
    constexpr int SH = V == 16 ? 1 : V == 8 ? 2 : V == 4 ? 3 : 4;   // 5 - log2(V)
    float v[V];
#pragma unroll
    for (int gi = 0; gi < NG; ++gi) {
        float s = 0.f, q = 0.f;
#pragma unroll
        for (int k = 0; k < W; ++k) {
            const float x = row_ok ? f[gi * W + k] : 0.f;
            s += x;
            q = fmaf(x, x, q);
        }
        v[2 * gi] = s;
        v[2 * gi + 1] = q;
    }
    const float total = halving_reduce<V>(v, lane);
    if ((lane & ((1 << SH) - 1)) == 0) {
        const int idx = lane >> SH;
        const int g = (n0 + (idx >> 1) * W) / CPG;
        atomicAdd(bins_b + 2 * g + (idx & 1), static_cast<unsigned long long>(__double2ll_rn(static_cast<double>(total) * scale)));
    }
}
LFM_DEVICE void gn_accumulate(const float* f, const GemmEpi& ep, int row, int M, int n0, int N, int lane) {
    if (n0 >= N) return;
    const int rep = static_cast<int>((blockIdx.x * 5u + (threadIdx.x >> 5)) % kGnBinReplicas);
    unsigned long long* bins_b = ep.gn_bins + (static_cast<size_t>((row < M ? row : M - 1) / ep.gn_hw) * kGnBinReplicas + rep) * 64;
    bins_b = reinterpret_cast<unsigned long long*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(bins_b), 0));
    const bool ok = row < M;
    const double sc = static_cast<double>(ep.gn_scale);
    switch (ep.gn_cpg) {
        case 4: gn_accumulate_chunk<4>(f, ok, n0, bins_b, lane, sc); break;
        case 8: gn_accumulate_chunk<8>(f, ok, n0, bins_b, lane, sc); break;
        case 16: gn_accumulate_chunk<16>(f, ok, n0, bins_b, lane, sc); break;
        case 32: gn_accumulate_chunk<32>(f, ok, n0, bins_b, lane, sc); break;
        case 64: gn_accumulate_chunk<64>(f, ok, n0, bins_b, lane, sc); break;
        default: break;
    }
}

// Write this lane's row segment (128 bytes = 8 x 16 B) into the warp's 32-row staging tile, 128B-swizzled
// (16-byte chunk j of row r lives at chunk j ^ (r & 7)): conflict-free, and the layout TMA expects.
LFM_DEVICE void stage_row_f32(uint8_t* stg, int lane, const float* f) {
    uint8_t* rowp = stg + lane * 128;
#pragma unroll
    for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(rowp + ((j ^ (lane & 7)) << 4)) = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
}
LFM_DEVICE void stage_row_bf16_half(uint8_t* stg, int lane, const float* f, int half) {  // 32 values -> chunks 4*half..
    uint8_t* rowp = stg + lane * 128;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 o;
        o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
        o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
        o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
        o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
        *reinterpret_cast<uint4*>(rowp + (((half * 4 + j) ^ (lane & 7)) << 4)) = o;
    }
}

// LayerNorm + adaLN modulate of `nrows` rows of the fp32 residual stream (just completed by the reduce-adds of this
// launch, so read through L2: ld.global.cg), executed by ONE finisher warp per 4-row unit: 2 rows in flight.
// Same arithmetic as ln_modulate_kernel (two-pass statistics in registers, eps 1e-6).
LFM_DEVICE void ln_finish_rows(const GemmEpi& ep, int row0, int nrows, int M, int D, int lane) {
    constexpr int MAXV = 9;  // D <= 1152
    const int nv = D / 128;
    const float* x = static_cast<const float*>(ep.out);
    const float inv_d = 1.0f / static_cast<float>(D);
    for (int r = row0; r < row0 + nrows; r += 2) {
        float4 v[2][MAXV];
        bool ok[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int row = r + u;
            ok[u] = row < M && row < row0 + nrows;
            const float4* xp = reinterpret_cast<const float4*>(x + static_cast<size_t>(ok[u] ? row : row0) * D);
#pragma unroll
            for (int m = 0; m < MAXV; ++m)
                if (m < nv) v[u][m] = __ldcg(xp + m * 32 + lane);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (!ok[u]) continue;  // warp-uniform
            const int row = r + u;
            float s = 0.f;
#pragma unroll
            for (int m = 0; m < MAXV; ++m)
                if (m < nv) s += (v[u][m].x + v[u][m].y) + (v[u][m].z + v[u][m].w);
            const float mean = warp_sum(s) * inv_d;
            float ss = 0.f;
#pragma unroll
            for (int m = 0; m < MAXV; ++m)
                if (m < nv) {
                    const float a = v[u][m].x - mean, b = v[u][m].y - mean, c = v[u][m].z - mean, d = v[u][m].w - mean;
                    ss += (a * a + b * b) + (c * c + d * d);
                }
            const float rstd = rsqrtf(warp_sum(ss) * inv_d + 1e-6f);
            const size_t boff = static_cast<size_t>(row / ep.rows_per_sample) * ep.ln_stride;
            const float4* shp = reinterpret_cast<const float4*>(ep.ln_shift + boff);
            const float4* scp = reinterpret_cast<const float4*>(ep.ln_scale + boff);
            uint2* yp = reinterpret_cast<uint2*>(ep.ln_out + static_cast<size_t>(row) * D);
#pragma unroll
            for (int m = 0; m < MAXV; ++m)
                if (m < nv) {
                    const float4 sh = __ldg(shp + m * 32 + lane), sc = __ldg(scp + m * 32 + lane);
                    const float a = fmaf((v[u][m].x - mean) * rstd, 1.f + sc.x, sh.x);
                    const float b = fmaf((v[u][m].y - mean) * rstd, 1.f + sc.y, sh.y);
                    const float c = fmaf((v[u][m].z - mean) * rstd, 1.f + sc.z, sh.z);
                    const float d = fmaf((v[u][m].w - mean) * rstd, 1.f + sc.w, sh.w);
                    yp[m * 32 + lane] = make_uint2(pack_bf16x2(a, b), pack_bf16x2(c, d));
                }
        }
    }
}

// bf16 output of one lane's 32-column row segment straight from registers (64 contiguous bytes, two full 32-byte
// sectors): no shared-memory staging, no TMA store - the pair kernel's mainloop already uses ~125 of the 128 B/clk of
// shared-memory bandwidth, and every staged byte (write + TMA read-back) extends the kernel (profiles/r2g_gemm2_epilogue_cost.md).
LFM_DEVICE void store_row_bf16_direct(__nv_bfloat16* rowp /* out + row * ldo + n0 */, const float* f, int n0, int N) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (n0 + 8 * j < N) {
            uint4 o;
            o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
            o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
            o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
            o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
            *reinterpret_cast<uint4*>(rowp + 8 * j) = o;
        }
    }
}

template <int EPI, bool FIN = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FIN ? kG2ThreadsFin : kG2Threads, 1)
gemm2_bf16_tcgen05(const __grid_constant__ CUtensorMap tmap_a,   // A [M, K], box {64, 128}
                   const __grid_constant__ CUtensorMap tmap_b,   // W [N, K], box {64, 128}
                   const __grid_constant__ CUtensorMap tmap_out, // out [M, ldo]: box {128 bytes, 32 rows}, 128B swizzle
                   const __grid_constant__ CUtensorMap tmap_bh,  // W [N, K], box {64, 64}: half-width tail tiles
                   int M, int N, int K, GemmEpi ep, ConvGeom cg, int allow_split, int ksplit, int split_row_pitch) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kG2Stages * kG2ABytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kG2Stages * kG2StageBytes);
    uint64_t* full_bar = bars;                        // [stages] (used in the leader CTA only)
    uint64_t* empty_bar = bars + kG2Stages;           // [stages] per CTA, signalled by the leader's multicast commit
    uint64_t* tmem_full = bars + 2 * kG2Stages;       // [2] per CTA, multicast commit
    uint64_t* tmem_empty = bars + 2 * kG2Stages + 2;  // [2] leader only: 16 epilogue warps (8 per CTA) arrive
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kG2Stages + 4);
    uint8_t* smem_stage = smem + kG2Stages * kG2StageBytes + 1024;  // 8 x 4 KB epilogue staging tiles (1024-aligned)
    constexpr int kFinUnits = 64;  // LayerNorm finisher: work units (of 4 rows) per 256-row block

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1;
    const int num_clusters = gridDim.x >> 1;

    const int n_blocks = (N + kG2BlockN - 1) / kG2BlockN;
    const int m_blocks = (M + 255) / 256;
    const int num_tiles = m_blocks * n_blocks;
    const int num_kb = K / 64;
    // Tail splitting: the tiles of the last, partially filled wave are cut into two 256 x 128 halves when that lets
    // them finish in half a wave (e.g. 256 tiles on 74 clusters: 3 waves + 34 tiles -> 3 waves + 68 half tiles).
    // Split-K (ksplit > 1; used when a GEMM has far fewer tiles than SM pairs, e.g. the 4x4 / 8x8 UNet layers):
    // work item = (tile, k-slice); every slice stores its fp32 partial tile into its own slab of a scratch buffer
    // (row offset slice * split_row_pitch in tmap_out) and a separate kernel adds the slabs in a fixed order.
    int full_count = num_tiles, num_items = num_tiles * ksplit;
    if (ksplit == 1) {
        const int rem = num_tiles % num_clusters;
        if (allow_split && num_tiles > num_clusters && rem > 0 && 2 * rem <= num_clusters) {
            full_count = num_tiles - rem;
            num_items = full_count + 2 * rem;
        } else if (allow_split == 2) {
            // tile-starved launch (the host sets 2 when 2 x tiles <= CTA pairs; small batches: 256 token rows give fc2 four tiles for
            // 74 CTA pairs): EVERY tile is cut into its two 256 x 128 halves, twice the SMs work and the serial K loop of an item takes
            // half the time.  Same accumulation order per element as the full-width tile: results are bit-identical.
            full_count = 0;
            num_items = 2 * num_tiles;
        }
    } else {
        full_count = num_items;
    }
    const int kb_per = (num_kb + ksplit - 1) / ksplit;
    auto decode = [&](int w, int& m_blk, int& n_blk, int& nh, int& width) {
        int tile = ksplit > 1 ? w / ksplit : w;
        nh = 0;
        width = kG2BlockN;
        if (w >= full_count) {
            tile = full_count + ((w - full_count) >> 1);
            nh = (w - full_count) & 1;
            width = kG2BlockN / 2;
        }
        m_blk = tile / n_blocks;
        n_blk = tile % n_blocks;
        if (ep.reverse_m) m_blk = m_blocks - 1 - m_blk;
    };

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_bh);
        prefetch_tmap(&tmap_a);
        prefetch_tmap(&tmap_b);
        prefetch_tmap(&tmap_out);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kG2Stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full[a], 1);
            mbar_init(&tmem_empty[a], 16);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc_2cta<512>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();  // barrier inits + TMEM allocation visible in both CTAs before any remote traffic
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();     // everything above overlapped the tail of the previous kernel; its outputs are complete from here on
    pdl_trigger();
    if (FIN && ep.fin_ctl != nullptr && blockIdx.x == 0 && warp == 3) {
        // prepare the control block of the NEXT finisher launch (the previous user of that block has completed)
        int* other = ep.fin_ctl + (ep.fin_set ^ 1) * ep.fin_stride;
        for (int i = lane; i < ep.fin_stride; i += 32) other[i] = i < 4 ? 0 : -1;
    }

    if (warp == 0) {
        // ===================== TMA producer (both CTAs) =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            // l2_keep (LFM_L2_HINT): the A operand of a residual GEMM is streamed once - mark it evict_first so that it does
            // not push the fp32 residual stream (re-read by the LayerNorm that follows) out of the L2
            const uint64_t a_policy = (EPI == EPI_GATE_RESID_F32 && ep.l2_keep) ? l2_policy_evict_first() : 0;
            for (int item = cluster_id; item < num_items; item += num_clusters) {
                int m_blk, n_blk, nh, width;
                decode(item, m_blk, n_blk, nh, width);
                const bool halfw = width != kG2BlockN;
                const int row_v = m_blk * 256 + static_cast<int>(rank) * 128;  // row of the output this CTA computes
                const int row_a = cg.a_mod > 0 ? row_v % cg.a_mod : row_v;
                const int row_b = (cg.batch_m > 0 ? (row_v / cg.batch_m) * cg.b_batch_rows : 0) + n_blk * kG2BlockN +
                                  nh * (kG2BlockN / 2) + static_cast<int>(rank) * (width / 2);
                const uint32_t tx_bytes = 2 * (kG2ABytes + (halfw ? kG2BBytes / 2 : kG2BBytes));
                int img0 = 0, h0 = 0, w0 = 0;
                if (cg.taps != 0) {
                    img0 = row_a / cg.HW;
                    h0 = (row_a % cg.HW) / cg.W;
                    w0 = row_a % cg.W;  // non-zero only when an image row is wider than the 128-pixel tile (W = 256, 512)
                }
                const int ks = ksplit > 1 ? item % ksplit : 0;
                const int kb0 = ks * kb_per, kb1 = min(num_kb, kb0 + kb_per);
                int tap = 0, cb = 0;
                if (cg.taps != 0) {
                    tap = kb0 / cg.cblocks;
                    cb = kb0 % cg.cblocks;
                }
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
                    if (cg.taps == 0) {
                        if (a_policy != 0)
                            tma_load_2d_2sm_hint(smem_a + stage * kG2ABytes, &tmap_a, &full_bar[stage], kb * 64, row_a, a_policy);
                        else
                            tma_load_2d_2sm(smem_a + stage * kG2ABytes, &tmap_a, &full_bar[stage], kb * 64, row_a);
                    } else {
                        const int r = tap / 3, sx = tap - 3 * r;
                        tma_load_4d_2sm(smem_a + stage * kG2ABytes, &tmap_a, &full_bar[stage], cb * 64, cg.stride * w0 + sx - 1,
                                        cg.stride * h0 + r - 1, img0);
                        if (++cb == cg.cblocks) {
                            cb = 0;
                            ++tap;
                        }
                    }
                    tma_load_2d_2sm(smem_b + stage * kG2BBytes, halfw ? &tmap_bh : &tmap_b, &full_bar[stage], kb * 64, row_b);
                    if (++stage == kG2Stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA, one thread) =====================
        if (rank == 0 && lane == 0) {
            constexpr uint32_t idesc_full = make_idesc_bf16(256, kG2BlockN, 0, 0);
            constexpr uint32_t idesc_half = make_idesc_bf16(256, kG2BlockN / 2, 0, 0);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int item = cluster_id; item < num_items; item += num_clusters) {
                const uint32_t idesc = item >= full_count ? idesc_half : idesc_full;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * kG2BlockN;
                const int ks = ksplit > 1 ? item % ksplit : 0;
                const int kb0 = ks * kb_per, kb1 = min(num_kb, kb0 + kb_per);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t da = make_smem_desc_sw128(smem_u32(smem_a + stage * kG2ABytes), 16, 1024);
                    const uint64_t db = make_smem_desc_sw128(smem_u32(smem_b + stage * kG2BBytes), 16, 1024);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_ss_2cta(tmem_d, da + 2 * k, db + 2 * k, idesc, ((kb - kb0) | k) != 0);
                    umma_commit_2cta(&empty_bar[stage]);
                    if (kb == kb1 - 1) umma_commit_2cta(&tmem_full[acc]);
                    if (++stage == kG2Stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                if (++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1;
                }
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ===================== epilogue: 8 warps, 128 rows x (2 x 128 columns) =====================
        // TMEM -> registers -> (bias / GELU / gate) -> swizzled smem staging tile -> TMA store, or TMA reduce-add
        // for the gated residual (x += g * (acc + b) is applied at L2: the SM never reads x).
        const int q = warp & 3;
        const int half = (warp - 4) >> 2;
        const uint64_t keep_policy = ep.l2_keep ? l2_policy_evict_last() : 0;
        uint8_t* stg0 = smem_stage + (warp - 4) * 4096;  // one staging tile per warp (measured: a second one at the
        constexpr int sbuf = 0;                           // cost of a pipeline stage does not pay)
        constexpr bool kBf16Out = (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_BF16);
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int item = cluster_id; item < num_items; item += num_clusters) {
            int m_blk, n_blk, nh, width;
            decode(item, m_blk, n_blk, nh, width);
            const int nch = width / 64;  // 32-column chunks per warp: 4 (full tile) or 2 (half-width tail tile)
            const int row_l = m_blk * 256 + static_cast<int>(rank) * 128 + q * 32;  // first row of this warp
            const int row = row_l + lane;
            const int row0 = row_l + (ksplit > 1 ? (item % ksplit) * split_row_pitch : 0);  // TMA row (slab of this k-slice)
            const int nbase = n_blk * kG2BlockN + nh * (kG2BlockN / 2) + half * (width / 2);
            const float* gate_row = nullptr;
            if (EPI == EPI_GATE_RESID_F32 && ep.gate != nullptr)  // gate == nullptr: plain residual add (gate 1)
                gate_row = ep.gate + static_cast<size_t>((row < M ? row : M - 1) / ep.rows_per_sample) * ep.gate_stride;
            const float* add_row = nullptr;
            if (EPI == EPI_BIAS_F32 && ep.addend != nullptr) add_row = ep.addend + static_cast<size_t>(row < M ? row : M - 1) * ep.ldo;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            if (ep.dbg_flags & 1) {  // measurement aid: mainloop speed without any TMEM drain (results are not written)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0);
                if (++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1;
                }
                continue;
            }
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kG2BlockN + half * (width / 2);
            uint32_t va[32], vb[32];
            float f[32];
            tmem_ld_32x32b_x32(taddr, va);
            const bool direct_bf16 = (ep.dbg_flags & 8) != 0;    // bf16 outputs: registers -> global, no staging (A/B switch)
            const bool dbg_no_math = (ep.dbg_flags & 2) != 0;    // measurement aid: TMEM is read, nothing else happens
            const bool dbg_no_store = (ep.dbg_flags & 4) != 0;   // measurement aid: everything but the global stores
#pragma unroll 1
            for (int c = 0; c < nch; c += 2) {
                tmem_ld_wait();
                tmem_ld_32x32b_x32(taddr + (c + 1) * 32, vb);
                if (dbg_no_math) {
                    tmem_ld_wait();
                    if (c + 2 < nch) tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
                    if (__uint_as_float(va[0] ^ vb[1]) == 1.2345e-31f) stg0[lane] = 1;  // keep the loads alive
                    continue;
                }
                epilogue_math<EPI>(va, f, ep, nbase + c * 32, N, gate_row, add_row);
                if ((EPI == EPI_BIAS_F32 || EPI == EPI_BIAS_BF16) && ep.gn_bins != nullptr) gn_accumulate(f, ep, row, M, nbase + c * 32, N, lane);
                // this staging tile is free once all but the most recent TMA op of this warp have READ their tile
                uint8_t* stg = stg0 + sbuf * 4096;
                if (kBf16Out && direct_bf16) {
                    if (row < M && ksplit == 1)
                        store_row_bf16_direct(static_cast<__nv_bfloat16*>(ep.out) + static_cast<size_t>(row) * ep.ldo + nbase + c * 32, f, nbase + c * 32, N);
                    tmem_ld_wait();
                    if (c + 2 < nch) tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
                    epilogue_math<EPI>(vb, f, ep, nbase + (c + 1) * 32, N, gate_row, add_row);
                    if (row < M && ksplit == 1)
                        store_row_bf16_direct(static_cast<__nv_bfloat16*>(ep.out) + static_cast<size_t>(row) * ep.ldo + nbase + (c + 1) * 32, f, nbase + (c + 1) * 32, N);
                    continue;
                }
                if (lane == 0) tma_store_wait_read<0>();
                __syncwarp();
                if (kBf16Out) {
                    stage_row_bf16_half(stg, lane, f, 0);
                } else {
                    stage_row_f32(stg, lane, f);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0 && nbase + c * 32 < N && !dbg_no_store) {
                        if (EPI == EPI_GATE_RESID_F32 && ep.l2_keep)
                            tma_reduce_add_2d_hint(&tmap_out, stg, nbase + c * 32, row0, keep_policy);
                        else if (EPI == EPI_GATE_RESID_F32)
                            tma_reduce_add_2d(&tmap_out, stg, nbase + c * 32, row0);
                        else
                            tma_store_2d(&tmap_out, stg, nbase + c * 32, row0);
                    }
                    if (lane == 0) tma_store_commit();
                }
                tmem_ld_wait();
                if (c + 2 < nch) tmem_ld_32x32b_x32(taddr + (c + 2) * 32, va);
                epilogue_math<EPI>(vb, f, ep, nbase + (c + 1) * 32, N, gate_row, add_row);
                if ((EPI == EPI_BIAS_F32 || EPI == EPI_BIAS_BF16) && ep.gn_bins != nullptr) gn_accumulate(f, ep, row, M, nbase + (c + 1) * 32, N, lane);
                if (kBf16Out) {
                    stage_row_bf16_half(stg, lane, f, 1);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0 && nbase + c * 32 < N && !dbg_no_store) tma_store_2d(&tmap_out, stg, nbase + c * 32, row0);  // 64 bf16 cols
                    if (lane == 0) tma_store_commit();
                } else {
                    stg = stg0 + sbuf * 4096;
                    if (lane == 0) tma_store_wait_read<0>();
                    __syncwarp();
                    stage_row_f32(stg, lane, f);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0 && nbase + (c + 1) * 32 < N && !dbg_no_store) {
                        if (EPI == EPI_GATE_RESID_F32 && ep.l2_keep)
                            tma_reduce_add_2d_hint(&tmap_out, stg, nbase + (c + 1) * 32, row0, keep_policy);
                        else if (EPI == EPI_GATE_RESID_F32)
                            tma_reduce_add_2d(&tmap_out, stg, nbase + (c + 1) * 32, row0);
                        else
                            tma_store_2d(&tmap_out, stg, nbase + (c + 1) * 32, row0);
                    }
                    if (lane == 0) tma_store_commit();
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0);  // leader's barrier
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1;
            }
            if (FIN && EPI == EPI_GATE_RESID_F32 && ep.ln_out != nullptr && lane == 0) {
                // this warp's share of the tile is in the residual stream once its reduce-adds have been performed
                tma_store_wait<0>();
                fence_proxy_async();
                __threadfence();                                             // release
                const int units = width == kG2BlockN ? 2 : 1;               // a half-width tail tile counts half
                const int old = atomicAdd(ep.rb_count + m_blk, units);
                if (old + units == 32 * n_blocks) {                          // 16 warps x 2 units x column tiles: block complete
                    atomicExch(ep.rb_count + m_blk, 0);                      // ready for the next launch
                    __threadfence();                                         // acquire
                    int* ctl = ep.fin_ctl + ep.fin_set * ep.fin_stride;
                    const int slot = atomicAdd(ctl + 1, 1);                  // reserve a queue slot, then publish the block index
                    atomicExch(ctl + 4 + slot, m_blk);
                }
            }
        }
        if (lane == 0) tma_store_wait<0>();  // all global writes of this warp are complete before the CTA exits
    } else if (FIN && warp >= 12) {
        // ===================== LayerNorm finisher: 4 warps per CTA pulling 4-row units from the global queue =====================
        if (ep.ln_out != nullptr) {
            int* ctl = ep.fin_ctl + ep.fin_set * ep.fin_stride;
            const int total_units = m_blocks * kFinUnits;
            for (;;) {
                int u = 0;
                if (lane == 0) u = atomicAdd(ctl, 1);
                u = __shfl_sync(0xffffffffu, u, 0);
                if (u >= total_units) break;
                const int q = u / kFinUnits, part = u % kFinUnits;
                int mb = 0;
                if (lane == 0) {
                    volatile int* vq = ctl + 4 + q;
                    while ((mb = *vq) < 0) __nanosleep(128);   // the q-th completed block has not been published yet
                }
                mb = __shfl_sync(0xffffffffu, mb, 0);
                __threadfence();                               // acquire: the rows of block mb are complete and visible
                ln_finish_rows(ep, mb * 256 + part * (256 / kFinUnits), 256 / kFinUnits, M, N, lane);
            }
        }
    }

    tc_fence_before();
    cluster_sync_all();  // nobody leaves while the peer may still read this CTA's smem / signal its barriers
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2cta<512>(tmem_base);
    }
}

}  // namespace lfm
