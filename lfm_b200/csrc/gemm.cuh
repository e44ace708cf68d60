// lfm_b200 - persistent, warp-specialised tcgen05 GEMM for the DiT linear layers.
//
//   C[M, N] = A[M, K] * W[N, K]^T   (A: activations bf16 row-major; W: nn.Linear weight, bf16, [out, in])
//
// Both operands are K-major, staged by TMA into 128B-swizzled shared memory (64-element K slabs), multiplied
// by tcgen05.mma.cta_group::1.kind::f16 (UMMA 128 x BLOCK_N x 16) into a double-buffered fp32 accumulator in
// TMEM, drained by 4 epilogue warps (tcgen05.ld 32x32b) that apply the fused epilogue and write to global.
//
// Warp roles (256 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator,
// warps 4..7 = epilogue (TMEM lane quadrant = warp % 4).
//
// Fused epilogues (reference ops they replace):
//   EPI_BIAS_BF16       out = bf16(acc + bias)                       attn.qkv       (timm Attention)
//   EPI_BIAS_GELU_BF16  out = bf16(gelu_tanh(acc + bias))            mlp.fc1 + act  (models/DiT.py:122-124)
//   EPI_GATE_RESID_F32  x  += gate[b] * (acc + bias)   (fp32 stream) attn.proj / mlp.fc2 + gated residual
//                                                                    (models/DiT.py:129-130)
//   EPI_BIAS_F32        out = acc + bias (fp32)                      all adaLN_modulation Linears in one GEMM
#pragma once
#include "common.cuh"

namespace lfm {

enum EpiMode { EPI_BIAS_BF16 = 0, EPI_BIAS_GELU_BF16 = 1, EPI_GATE_RESID_F32 = 2, EPI_BIAS_F32 = 3 };

struct GemmEpi {
    const float* bias;    // [N] or nullptr
    void* out;            // bf16 [M, ldo] / fp32 [M, ldo]; for EPI_GATE_RESID_F32 the residual stream (read+write)
    int ldo;              // row pitch of out, elements
    const float* gate;    // EPI_GATE_RESID_F32: gate[b * gate_stride + n]
    int gate_stride;      // elements between samples in the modulation table
    int rows_per_sample;  // tokens per sample (b = row / rows_per_sample)
    // Optional (pair kernel, EPI_BIAS_F32): GroupNorm statistics of the OUTPUT accumulated in the epilogue -
    // bins[((row / gn_hw) * kGnBinReplicas + r) * 64 + 2 g + {0,1}] += {sum, sum of squares} of group g = column / gn_cpg, as
    // gn_scale fixed point (integer atomics => the result does not depend on the order of arrival: deterministic).  r is any of
    // kGnBinReplicas copies (chosen per warp; the consumer adds them up - integers, so still exact): persistent CTAs walk the
    // tiles of ONE image together, and with a single copy every atomic of the chip queued on the same four 128-byte lines
    // (a 128-channel 256 x 256 VAE layer: 2.1 M atomics, +525 us on a 410 us convolution; profiles/r2l_vae_launches.md).
    unsigned long long* gn_bins = nullptr;
    int gn_cpg = 0;
    int gn_hw = 1;
    float gn_scale = 268435456.0f;  // fixed-point scale of this statistics slot (gn_fix_scale); the consumer reads GnApplyArgs::bins_unit
    // Pair kernel: walk the M blocks from the last to the first.  Consecutive kernels of a network alternate
    // direction so that each one starts on the rows its producer touched LAST - the part still resident in L2.
    int reverse_m = 0;
    // Pair kernel, EPI_GATE_RESID_F32: the TMA reduce-add into the residual stream carries the evict_last L2 policy.
    int l2_keep = 0;
    // Pair kernel, EPI_BIAS_F32: out = addend + acc + bias, the residual connection of a convolutional block added by
    // the SM (fp32 [M, ldo]; may alias out) - so that the block's OUTPUT statistics (gn_bins) can be taken in the same
    // epilogue, which a reduce-add performed at L2 never sees.
    const float* addend = nullptr;
    int dbg_flags = 0;  // measurement aids (LFM_G2_DBG, profiles/r2g_gemm2_epilogue_cost.md): 1 accumulators released undrained,
                        // 2 TMEM reads only, 4 no global stores, 8 bf16 rows stored straight from registers
    // Pair kernel with the LayerNorm finisher (gemm2_bf16_tcgen05<EPI_GATE_RESID_F32, true>; N == ldo == D): once every
    // column tile of a 256-row block of the residual stream has been added, the block is published in a GLOBAL queue and
    // the finisher warps of ALL CTAs pull 4-row units from it (ticket counter) and produce the NEXT layer's operand
    // ln_out = LayerNorm(x) * (1 + ln_scale) + ln_shift (bf16; models/DiT.py:20-21, 129-130) while the rows are still in
    // L2 - the stand-alone LayerNorm pass over x disappears.  (Round 2's first version let the CTA that arrived last do the
    // whole block: 2.6x slower end to end.)  rb_count[m_blk] counts arrivals (zero on entry; reset by the last arriver).
    // fin_ctl: two control blocks of fin_stride ints {ticket, tail, -, -, queue[m_blocks]}; a launch uses block fin_set and
    // re-initialises the OTHER one for the finisher launch after it (they alternate 0 / 1 within a network evaluation).
    int* rb_count = nullptr;
    int* fin_ctl = nullptr;
    int fin_stride = 0;
    int fin_set = 0;
    __nv_bfloat16* ln_out = nullptr;  // nullptr: this launch only keeps the control blocks alternating
    const float* ln_shift = nullptr;  // [sample * ln_stride + column]
    const float* ln_scale = nullptr;
    int ln_stride = 0;
};
constexpr int kGnBinReplicas = 16;
// Fixed-point scale of the fused GroupNorm statistics, chosen per slot from n = H * W * C / 32, the elements of one
// (image, group).  The replicas are added as long long, so the sum of squares n * E[x^2] must stay below 2^63 / scale:
// 2^28 (every layer with n <= 2^19 - all of the 256-pixel decode and the UNets) allows an rms of 2^17.5 / sqrt(n), 256 at
// n = 2^19, 181 at 2^20.  The 512-pixel decode's last stage reaches n = 2^20 (2^21 with LFM_UNET_FUSE_OUT=1): 2^22 there,
// rms up to 1448 / 1024.  One atomic rounds by at most 0.5 / scale (2^-23 at 2^22): negligible next to sums of 2^20 values.
constexpr double kGnFixScale = 268435456.0;   // 2^28
constexpr double kGnFixScaleWide = 4194304.0; // 2^22
constexpr long long kGnFixWideN = 1 << 19;    // n above which a slot uses kGnFixScaleWide
constexpr double kGnMinRms = 256.0;           // the host refuses a slot whose scale allows a smaller rms than this
__host__ __device__ constexpr double gn_fix_scale(long long n) { return n <= kGnFixWideN ? kGnFixScale : kGnFixScaleWide; }

constexpr int kGemmBlockM = 128;
constexpr int kGemmBlockK = 64;  // 64 bf16 = one 128-byte swizzle row
constexpr int kGemmThreads = 256;

template <int BLOCK_N>
struct GemmCfg {
    static constexpr int kABytes = kGemmBlockM * kGemmBlockK * 2;
    static constexpr int kBBytes = BLOCK_N * kGemmBlockK * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kStages = (BLOCK_N == 256) ? 4 : 6;
    static constexpr int kTmemCols = 2 * BLOCK_N;  // double-buffered accumulator
    static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BLOCK_N, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int M, int N,
                  int K, GemmEpi ep) {
    using Cfg = GemmCfg<BLOCK_N>;
    constexpr int kStages = Cfg::kStages;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kStages * Cfg::kABytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
    uint64_t* full_bar = bars;                    // [kStages] TMA -> MMA
    uint64_t* empty_bar = bars + kStages;         // [kStages] MMA -> TMA
    uint64_t* tmem_full = bars + 2 * kStages;     // [2] MMA -> epilogue
    uint64_t* tmem_empty = bars + 2 * kStages + 2;  // [2] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    const int n_blocks = (N + BLOCK_N - 1) / BLOCK_N;
    const int m_blocks = (M + kGemmBlockM - 1) / kGemmBlockM;
    const int num_tiles = m_blocks * n_blocks;
    const int num_kb = K / kGemmBlockK;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_a);
        prefetch_tmap(&tmap_b);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full[a], 1);
            mbar_init(&tmem_empty[a], 128);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();
    pdl_trigger();

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int m_blk = tile / n_blocks, n_blk = tile % n_blocks;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                    tma_load_2d(smem_a + stage * Cfg::kABytes, &tmap_a, &full_bar[stage], kb * kGemmBlockK,
                                m_blk * kGemmBlockM);
                    tma_load_2d(smem_b + stage * Cfg::kBBytes, &tmap_b, &full_bar[stage], kb * kGemmBlockK,
                                n_blk * BLOCK_N);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (one thread) =====================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(kGemmBlockM, BLOCK_N, 0, 0);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t da = make_smem_desc_sw128(smem_u32(smem_a + stage * Cfg::kABytes), 16, 1024);
                    const uint64_t db = make_smem_desc_sw128(smem_u32(smem_b + stage * Cfg::kBBytes), 16, 1024);
#pragma unroll
                    for (int k = 0; k < kGemmBlockK / 16; ++k) {
                        // +32 bytes per UMMA_K step inside the 128B swizzle row => +2 in the (addr >> 4) field
                        umma_ss(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    }
                    umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
                    if (kb == num_kb - 1) umma_commit(&tmem_full[acc]);
                    if (++stage == kStages) {
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
    } else if (warp >= 4) {
        // ===================== epilogue (4 warps, one TMEM lane quadrant each) =====================
        const int q = warp & 3;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int m_blk = tile / n_blocks, n_blk = tile % n_blocks;
            const int row = m_blk * kGemmBlockM + q * 32 + lane;
            const bool row_ok = row < M;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
            const float* gate_row = nullptr;
            if (EPI == EPI_GATE_RESID_F32 && row_ok)
                gate_row = ep.gate + static_cast<size_t>(row / ep.rows_per_sample) * ep.gate_stride;
#pragma unroll 1
            for (int c = 0; c < BLOCK_N / 32; ++c) {
                const int n0 = n_blk * BLOCK_N + c * 32;
                uint32_t v[32];
                float4 xr[8];
                if (EPI == EPI_GATE_RESID_F32) {
                    const float4* xp = reinterpret_cast<const float4*>(static_cast<float*>(ep.out) +
                                                                       static_cast<size_t>(row) * ep.ldo + n0);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (row_ok && n0 + j * 4 < N) xr[j] = xp[j];
                }
                tmem_ld_32x32b_x32(taddr + c * 32, v);
                tmem_ld_wait();
                if (n0 >= N) continue;
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                if (ep.bias != nullptr) {
                    const float4* bp = reinterpret_cast<const float4*>(ep.bias + n0);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (n0 + j * 4 < N) {
                            const float4 b4 = __ldg(bp + j);
                            f[4 * j + 0] += b4.x;
                            f[4 * j + 1] += b4.y;
                            f[4 * j + 2] += b4.z;
                            f[4 * j + 3] += b4.w;
                        }
                    }
                }
                if (EPI == EPI_BIAS_GELU_BF16) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = gelu_tanh(f[j]);
                }
                // NOTE: no divergent `continue` here - the next tcgen05.ld is .sync.aligned (whole warp).
                if (!row_ok) {
                    // rows beyond M (TMA zero-filled): nothing to store
                } else if (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_BF16) {
                    uint4* op = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(ep.out) +
                                                         static_cast<size_t>(row) * ep.ldo + n0);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (n0 + j * 8 < N) {
                            uint4 o;
                            o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
                            o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
                            o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
                            o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
                            op[j] = o;
                        }
                    }
                } else if (EPI == EPI_BIAS_F32) {
                    float4* op =
                        reinterpret_cast<float4*>(static_cast<float*>(ep.out) + static_cast<size_t>(row) * ep.ldo + n0);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (n0 + j * 4 < N) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                } else {  // EPI_GATE_RESID_F32
                    float4* op =
                        reinterpret_cast<float4*>(static_cast<float*>(ep.out) + static_cast<size_t>(row) * ep.ldo + n0);
                    const float4* gp = reinterpret_cast<const float4*>(gate_row + n0);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (n0 + j * 4 < N) {
                            const float4 g4 = __ldg(gp + j);
                            float4 x4 = xr[j];
                            x4.x = fmaf(g4.x, f[4 * j + 0], x4.x);
                            x4.y = fmaf(g4.y, f[4 * j + 1], x4.y);
                            x4.z = fmaf(g4.z, f[4 * j + 2], x4.z);
                            x4.w = fmaf(g4.w, f[4 * j + 3], x4.w);
                            op[j] = x4;
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

}  // namespace lfm
