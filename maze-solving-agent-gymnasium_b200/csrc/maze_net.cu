// DQN / DDQN network on the B200 tensor cores (sm_100a): forward, double-Q target, backward and AdamW of
// the net of agents/ddqn_agent.py:18-52 (conv 3->32 3x3 pad 1, LeakyReLU, MaxPool 2 -> 1568 (+6) -> 1024
// -> 512 -> 4) and its update agents/ddqn_agent.py:113-152 (double-Q target, MSE, gradient clamp +-1, AdamW),
// reading the replay ring's bit-packed windows directly (csrc/maze_dqn.cu).  The net's Dropout (p = 0.2 in the
// reference, active because the reference never calls eval()) runs in the conv epilogue when maze_dqn_net.dropout > 0
// (mask stream: include/maze_b200.h); maze_dqn_net.update = 1 swaps the double-Q target for the plain DQN max target of
// agents/dqn_agent.py.
//
// Dense contractions run as tcgen05.mma (bf16 x bf16 -> fp32 in TMEM), operands staged by TMA:
//   net_gemm_kernel   C[M,N] = A[M,K] . B[N,K]^T, both operands K-major bf16, 128 x BN x 64 tiles, SWIZZLE_128B,
//                     4-6 stage TMA ring, one MMA-issuing thread, 4 epilogue warps reading TMEM; epilogues:
//                     bias + activation (forward), activation-derivative mask (backward data), fp32 red.add
//                     with split-K (weight gradients)
//   net_features_kernel  the 3x3 convolution as an implicit GEMM: per sample a [(row, col16), (channel, dx)]
//                     bf16 image matrix in shared memory, three accumulating MMAs per 128-position tile whose
//                     A descriptors start 16 rows apart (dy = -1, 0, +1), bias + 2x2 max-pool + LeakyReLU in the
//                     TMEM epilogue
// Everything else (fc3 head, loss, conv weight gradient, transposes, AdamW) is CUDA-core work: < 2 % of the FLOPs.
#include <cstdio>
#include <cstring>
#include "maze_common.cuh"
#include "maze_replay.cuh"
#include "maze_tc.cuh"

namespace {

typedef __nv_bfloat16 bf16;

constexpr int BM = 128, BK = 64;
constexpr int GEMM_THREADS = 192;

enum { EPI_BIAS_ACT = 0, EPI_MASK = 1, EPI_RED_F32 = 2 };
enum { ACT_NONE = 0, ACT_LRELU = 1, ACT_RELU = 2 };
constexpr float LRELU_SLOPE = 0.01f;   // nn.LeakyReLU() default (ddqn_agent.py:28,38)

struct GemmArgs {
    int M, N, K;          // C[M, N] = A[M, K] . B[N, K]^T
    void* C;              // bf16 (EPI_BIAS_ACT, EPI_MASK) or fp32 accumulators (EPI_RED_F32)
    int ldc;
    const float* bias;    // [N] or null                       (EPI_BIAS_ACT)
    const bf16* aux;      // forward activation [M, ldaux]     (EPI_MASK: derivative of `act` taken at it)
    int ldaux;
    int act;
    int splits;           // CTAs along K per output tile (EPI_RED_F32)
};

template <int BN>
struct GemmCfg {
    static constexpr int STAGES = BN == 256 ? 4 : 6;
    static constexpr uint32_t A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024;   // + slack for the 1024-byte alignment
};

// MN == false: A [M, K] and B [N, K] row-major (K-major operands: one TMA box of BM (BN) rows x 64 K-elements per stage,
//              8-row x 128-byte swizzle atoms 1024 bytes apart along M / N).
// MN == true:  A [K, M] and B [K, N] row-major, i.e. C = A^T . B -- the weight gradients contract over the batch, and
//              the activations are stored [batch, features].  MN-major operands: per stage BM / 64 (BN / 64) TMA boxes
//              of 64 K-rows x 64 M (N)-elements; inside a box the 8-row swizzle atoms follow each other along K
//              (stride-dimension offset 1024), the boxes along M / N (leading-dimension offset 8192); one UMMA of
//              K = 16 starts 16 rows = 2048 bytes further.  No transposed copies of the activations are needed.
// The bf16 epilogues of one accumulator tile for one warp (32 rows; lane = row; 32 columns per TMEM load).  The main loop
// saturates L2 -> SM bandwidth, so a global load issued from here waits microseconds, and a store of one 16-byte piece per
// lane touches 32 lines per instruction.  Hence: the bias slice of the tile is staged in shared memory by the caller
// (`sb`, zero beyond N, or nullptr); the stored activations of EPI_MASK are fetched one 32-column chunk ahead of their
// use; and the output leaves through a TMA store -- 64 columns x 32 rows are packed to bf16, written to the warp's own
// 4 KB staging tile in the 128-byte swizzle the tensor map expects (conflict-free: lane r writes piece p at p ^ (r & 7)),
// and one lane issues cp.async.bulk.tensor (rows >= M / columns >= N are clipped by the TMA unit).
// (Per-element __ldg of the bias: fc1 forward 90 us instead of 50; per-lane 16-byte stores: fc2 backward-data 25 us.)
template <int EPI, int BN>
__device__ __forceinline__ void epi_bf16_tile(const GemmArgs& g, const CUtensorMap* tmC, uint32_t taddr, int row0, int lane, int n0, const float* sb,
                                              uint8_t* stage) {
    const int row = row0 + lane;
    const bool row_ok = row < g.M;
    const bf16* arow = g.aux + (size_t)row * g.ldaux + n0;
    const float neg = g.act == ACT_LRELU ? LRELU_SLOPE : 0.f;
    uint4 h[4], hn[4];
    auto load_aux = [&](uint4 (&dst)[4], int c0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            dst[u] = make_uint4(0, 0, 0, 0);
            if (row_ok && n0 + c0 + 8 * u + 8 <= g.N) dst[u] = __ldg(reinterpret_cast<const uint4*>(arow + c0 + 8 * u));
        }
    };
    if constexpr (EPI == EPI_MASK) load_aux(h, 0);
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 64) {
        if (n0 + c0 >= g.N) break;
        uint32_t packed[32];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int cc = c0 + 32 * half;
            uint32_t v[32];
            tc::tmem_ld32(taddr + (uint32_t)cc, v);
            if constexpr (EPI == EPI_MASK) {
                if (cc + 32 < BN) load_aux(hn, cc + 32);
            }
            tc::tmem_ld_wait();
            if constexpr (EPI == EPI_BIAS_ACT) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (sb) b = *reinterpret_cast<const float4*>(sb + cc + j);
                    float x[4] = {__uint_as_float(v[j]) + b.x, __uint_as_float(v[j + 1]) + b.y, __uint_as_float(v[j + 2]) + b.z, __uint_as_float(v[j + 3]) + b.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (g.act == ACT_LRELU) x[u] = x[u] > 0.f ? x[u] : LRELU_SLOPE * x[u];
                        else if (g.act == ACT_RELU) x[u] = fmaxf(x[u], 0.f);
                    }
                    packed[16 * half + (j >> 1)] = tc::pack_bf16x2(x[0], x[1]);
                    packed[16 * half + (j >> 1) + 1] = tc::pack_bf16x2(x[2], x[3]);
                }
            } else {   // EPI_MASK: dL/d(pre-activation) = dL/d(activation) * act'(pre), sign taken from the stored activation
#pragma unroll
                for (int u8 = 0; u8 < 4; ++u8) {
                    const uint32_t hw[4] = {h[u8].x, h[u8].y, h[u8].z, h[u8].w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        // bf16 sign/zero test on the raw bits: > 0 <=> sign clear and magnitude non-zero
                        const uint32_t lo = hw[u] & 0xffffu, hi = hw[u] >> 16;
                        const float f0 = (lo != 0 && lo < 0x8000u) ? 1.f : neg, f1 = (hi != 0 && hi < 0x8000u) ? 1.f : neg;
                        packed[16 * half + 4 * u8 + u] = tc::pack_bf16x2(__uint_as_float(v[8 * u8 + 2 * u]) * f0, __uint_as_float(v[8 * u8 + 2 * u + 1]) * f1);
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) h[u] = hn[u];
            }
        }
        if (lane == 0) tc::tma_store_wait_read();   // the previous store has read the staging tile
        __syncwarp();
#pragma unroll
        for (int pc = 0; pc < 8; ++pc)
            *reinterpret_cast<uint4*>(stage + lane * 128 + ((pc ^ (lane & 7)) << 4)) = make_uint4(packed[4 * pc], packed[4 * pc + 1], packed[4 * pc + 2], packed[4 * pc + 3]);
        tc::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
            tc::tma_store_2d(tmC, tc::smem_u32(stage), n0 + c0, row0);
            tc::tma_store_commit();
        }
    }
}

// The tile's slice of the bias vector -> shared memory, by the four epilogue warps (128 threads, named barrier 1).  Two
// buffers, indexed like the accumulator stages: a warp can be at most one tile ahead of the slowest one.
template <int BN>
__device__ __forceinline__ void stage_bias(const GemmArgs& g, float* sb, int n0, int et) {
    for (int i = et; i < BN; i += 128) sb[i] = n0 + i < g.N ? __ldg(g.bias + n0 + i) : 0.f;
    asm volatile("bar.sync 1, 128;" ::: "memory");
}

template <int BN, int EPI, bool MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
net_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                const GemmArgs g) {
    using Cfg = GemmCfg<BN>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr uint32_t ACC_COLS = 2 * BN;   // two accumulator stages: the epilogue of tile i overlaps the main loop of tile i + 1
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bars[2 * STAGES + 4];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[2][BN];   // the tile's bias slice, per accumulator stage
    __shared__ __align__(1024) uint8_t s_stage[EPI == EPI_RED_F32 ? 1 : 4][EPI == EPI_RED_F32 ? 1024 : 4096];   // per epilogue warp: 32 rows x 64 bf16, swizzled
    const uint32_t base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B atoms are 1024-byte aligned
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Persistent CTA: tiles blockIdx.x, blockIdx.x + gridDim.x, ...; tile t = (split, n block, m block) with the m block
    // fastest, so CTAs that run side by side share their B (weight) tile in L2.
    const int tiles_m = (g.M + BM - 1) / BM, tiles_n = (g.N + BN - 1) / BN, splits = g.splits;
    const int num_tiles = tiles_m * tiles_n * splits;
    const int nkb_total = (g.K + BK - 1) / BK;
    const uint32_t full0 = tc::smem_u32(&bars[0]), empty0 = tc::smem_u32(&bars[STAGES]);
    const uint32_t acc_full0 = tc::smem_u32(&bars[2 * STAGES]), acc_empty0 = tc::smem_u32(&bars[2 * STAGES + 2]);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA);
        tc::tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(full0 + 8 * s, 1);
            tc::mbar_init(empty0 + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(acc_full0 + 8 * a, 1);    // one tcgen05.commit
            tc::mbar_init(acc_empty0 + 8 * a, 4);   // one arrival per epilogue warp
        }
        tc::mbar_fence_init();
    }
    if (warp == 1) {
        tc::tmem_alloc(tc::smem_u32(&tmem_slot), ACC_COLS);
        tc::tmem_relinquish();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    auto tile_coords = [&](int t, int& m0, int& n0, int& kb_begin, int& nkb) {
        const int mb = t % tiles_m, rest = t / tiles_m;
        const int nb = rest % tiles_n, sp = rest / tiles_n;
        m0 = mb * BM;
        n0 = nb * BN;
        kb_begin = (int)((long long)nkb_total * sp / splits);
        nkb = (int)((long long)nkb_total * (sp + 1) / splits) - kb_begin;   // >= 1: the launcher keeps splits <= k-blocks
    };

    if (warp == 0) {
        if (lane == 0) {   // TMA producer
            uint32_t it = 0;   // k-block counter over all tiles of this CTA: ring position and phase
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                int m0, n0, kb_begin, nkb;
                tile_coords(t, m0, n0, kb_begin, nkb);
                for (int i = 0; i < nkb; ++i, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                    tc::mbar_wait(empty0 + 8 * s, ph ^ 1u);
                    tc::mbar_expect_tx(full0 + 8 * s, Cfg::STAGE_BYTES);
                    const uint32_t a_dst = base + s * Cfg::STAGE_BYTES;
                    if constexpr (!MN) {
                        tc::tma_load_2d(a_dst, &tmA, full0 + 8 * s, (kb_begin + i) * BK, m0);
                        tc::tma_load_2d(a_dst + Cfg::A_BYTES, &tmB, full0 + 8 * s, (kb_begin + i) * BK, n0);
                    } else {
#pragma unroll
                        for (int j = 0; j < BM / 64; ++j) tc::tma_load_2d(a_dst + j * 8192, &tmA, full0 + 8 * s, m0 + 64 * j, (kb_begin + i) * BK);
#pragma unroll
                        for (int j = 0; j < BN / 64; ++j)
                            tc::tma_load_2d(a_dst + Cfg::A_BYTES + j * 8192, &tmB, full0 + 8 * s, n0 + 64 * j, (kb_begin + i) * BK);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // MMA issuer
            constexpr uint32_t idesc = tc::idesc_bf16(BM, BN) | (MN ? (1u << 15) | (1u << 16) : 0u);   // bits 15 / 16: A / B are MN-major
            uint32_t it = 0, local = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++local) {
                int m0, n0, kb_begin, nkb;
                tile_coords(t, m0, n0, kb_begin, nkb);
                const uint32_t acc = local & 1u;
                tc::mbar_wait(acc_empty0 + 8 * acc, ((local >> 1) & 1u) ^ 1u);   // the epilogue has drained this accumulator stage
                tc::tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int i = 0; i < nkb; ++i, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                    tc::mbar_wait(full0 + 8 * s, ph);
                    tc::tc_fence_after();
                    const uint32_t a_addr = base + s * Cfg::STAGE_BYTES;
                    const uint64_t da = tc::smem_desc(a_addr, MN ? 8192 : 0, 1024, tc::SWIZZLE_128B);
                    const uint64_t db = tc::smem_desc(a_addr + Cfg::A_BYTES, MN ? 8192 : 0, 1024, tc::SWIZZLE_128B);
                    // next UMMA (K = 16): K-major 32 bytes further inside the 128-byte swizzle row, MN-major 16 rows = 2048 bytes further
                    constexpr uint32_t kstep = MN ? (2048u >> 4) : (32u >> 4);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k)
                        tc::umma_bf16(tmem_d, da + kstep * k, db + kstep * k, idesc, (uint32_t)((i | k) != 0));
                    tc::umma_commit(empty0 + 8 * s);   // frees the stage once these MMAs have read it
                }
                tc::umma_commit(acc_full0 + 8 * acc);
            }
        }
    } else {   // epilogue: warp w may read TMEM lanes 32 (w % 4) .. + 31
        const int q = warp & 3;
        const bool has_bias = EPI == EPI_BIAS_ACT && g.bias != nullptr;
        uint32_t local = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++local) {
            int m0, n0, kb_begin, nkb;
            tile_coords(t, m0, n0, kb_begin, nkb);
            const uint32_t acc = local & 1u;
            if (has_bias) stage_bias<BN>(g, s_bias[acc], n0, (warp - 2) * 32 + lane);   // overlaps the tile's main loop
            tc::mbar_wait(acc_full0 + 8 * acc, (local >> 1) & 1u);
            tc::tc_fence_after();
            const int row = m0 + q * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
            if constexpr (EPI == EPI_RED_F32) {
                const bool row_ok = row < g.M;
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    if (n0 + c0 >= g.N) break;
                    uint32_t v[32];
                    tc::tmem_ld32(taddr + (uint32_t)c0, v);
                    tc::tmem_ld_wait();
                    const int col0 = n0 + c0;
                    float* dst = reinterpret_cast<float*>(g.C) + (size_t)row * g.ldc + col0;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (row_ok && col0 + j + 4 <= g.N)
                            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(__uint_as_float(v[j])),
                                         "f"(__uint_as_float(v[j + 1])), "f"(__uint_as_float(v[j + 2])), "f"(__uint_as_float(v[j + 3]))
                                         : "memory");
                    }
                }
            } else {
                epi_bf16_tile<EPI, BN>(g, &tmC, taddr, m0 + q * 32, lane, n0, has_bias ? s_bias[acc] : nullptr, s_stage[warp - 2]);
            }
            // every value of this accumulator stage is in registers: hand the stage back to the MMA issuer
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(acc_empty0 + 8 * acc);
        }
        if (EPI != EPI_RED_F32 && lane == 0) tc::tma_store_wait_all();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem_base, ACC_COLS);
}

// ------------------------------------------------------------------------------------------------------
// The same GEMM on CTA PAIRS (tcgen05 cta_group::2): two CTAs of a cluster, on the two SMs of a TPC, compute one
// 256 x 256 output tile.  Each CTA loads its own 128 rows of A and HALF of the B tile (128 of the 256 N rows); the leader
// CTA's MMA thread issues tcgen05.mma.cta_group::2 (M = 256), which reads both CTAs' shared memory and writes each CTA's
// 128 rows of the accumulator into that CTA's own TMEM.  Per 128 x 256 outputs an SM now pulls 32 KB per k-block from L2
// instead of 48 KB: the single-CTA kernel is bound by L2 -> SM bandwidth once its operands are not L2-warm (ncu
// profiles/r02r: 630 MB through the crossbar in 90 us, tensor pipe 33 %).  Protocol: the "full" barrier of a stage lives
// in the leader (it expects the bytes of both CTAs; both CTAs' TMA loads complete on it through its shared::cluster
// address); "empty" and "accumulator full" barriers exist in both CTAs and are released by multicast tcgen05.commit;
// "accumulator empty" lives in the leader and collects the arrivals of all eight epilogue warps of the pair.
// K-major operands, BN = 256, no split-K (the forward and backward-data GEMMs).
constexpr int PAIR_STAGES = 6;
constexpr uint32_t PAIR_A_BYTES = 128 * BK * 2, PAIR_B_BYTES = 128 * BK * 2, PAIR_STAGE_BYTES = PAIR_A_BYTES + PAIR_B_BYTES;
constexpr size_t PAIR_SMEM = (size_t)PAIR_STAGES * PAIR_STAGE_BYTES + 1024;

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
net_gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                     const GemmArgs g) {
    constexpr int BN = 256;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bars[2 * PAIR_STAGES + 4];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[2][BN];
    __shared__ __align__(1024) uint8_t s_stage[4][4096];
    const uint32_t base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
    const int tiles_m = (g.M + 255) / 256, tiles_n = (g.N + BN - 1) / BN;
    const int num_tiles = tiles_m * tiles_n;
    const int nkb = (g.K + BK - 1) / BK;
    const uint32_t full0 = tc::smem_u32(&bars[0]), empty0 = tc::smem_u32(&bars[PAIR_STAGES]);
    const uint32_t acc_full0 = tc::smem_u32(&bars[2 * PAIR_STAGES]), acc_empty0 = tc::smem_u32(&bars[2 * PAIR_STAGES + 2]);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA);
        tc::tma_prefetch_desc(&tmB);
        for (int s = 0; s < PAIR_STAGES; ++s) {
            tc::mbar_init(full0 + 8 * s, 1);
            tc::mbar_init(empty0 + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(acc_full0 + 8 * a, 1);
            tc::mbar_init(acc_empty0 + 8 * a, 8);   // four epilogue warps in each CTA of the pair
        }
        tc::mbar_fence_init();
    }
    if (warp == 1) {
        tc::tmem_alloc_pair(tc::smem_u32(&tmem_slot), 512);
        tc::tmem_relinquish_pair();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync();   // both CTAs' barriers are initialised before anything arrives on them from the peer
    tc::tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {   // TMA producer (both CTAs)
            uint32_t it = 0;
            for (int t = pair; t < num_tiles; t += num_pairs) {
                const int m0 = (t % tiles_m) * 256 + (int)rank * 128, n0 = (t / tiles_m) * BN + (int)rank * 128;
                for (int i = 0; i < nkb; ++i, ++it) {
                    const uint32_t s = it % PAIR_STAGES, ph = (it / PAIR_STAGES) & 1u;
                    tc::mbar_wait(empty0 + 8 * s, ph ^ 1u);
                    if (leader) tc::mbar_expect_tx(full0 + 8 * s, 2 * PAIR_STAGE_BYTES);
                    const uint32_t full_leader = tc::mapa(full0 + 8 * s, 0);
                    const uint32_t a_dst = base + s * PAIR_STAGE_BYTES;
                    tc::tma_load_2d_pair(a_dst, &tmA, full_leader, i * BK, m0);
                    tc::tma_load_2d_pair(a_dst + PAIR_A_BYTES, &tmB, full_leader, i * BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {   // MMA issuer: the leader CTA only
            constexpr uint32_t idesc = tc::idesc_bf16(256, BN);
            uint32_t it = 0, local = 0;
            for (int t = pair; t < num_tiles; t += num_pairs, ++local) {
                const uint32_t acc = local & 1u;
                tc::mbar_wait(acc_empty0 + 8 * acc, ((local >> 1) & 1u) ^ 1u);
                tc::tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int i = 0; i < nkb; ++i, ++it) {
                    const uint32_t s = it % PAIR_STAGES, ph = (it / PAIR_STAGES) & 1u;
                    tc::mbar_wait(full0 + 8 * s, ph);
                    tc::tc_fence_after();
                    const uint32_t a_addr = base + s * PAIR_STAGE_BYTES;
                    const uint64_t da = tc::smem_desc(a_addr, 0, 1024, tc::SWIZZLE_128B);
                    const uint64_t db = tc::smem_desc(a_addr + PAIR_A_BYTES, 0, 1024, tc::SWIZZLE_128B);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) tc::umma_bf16_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, (uint32_t)((i | k) != 0));
                    tc::umma_commit_pair(empty0 + 8 * s, 3);   // frees the stage in both CTAs
                }
                tc::umma_commit_pair(acc_full0 + 8 * acc, 3);
            }
        }
    } else {   // epilogue (both CTAs): this CTA's 128 rows of the tile
        const int q = warp & 3;
        const bool has_bias = EPI == EPI_BIAS_ACT && g.bias != nullptr;
        uint32_t local = 0;
        for (int t = pair; t < num_tiles; t += num_pairs, ++local) {
            const int m0 = (t % tiles_m) * 256 + (int)rank * 128, n0 = (t / tiles_m) * BN;
            const uint32_t acc = local & 1u;
            if (has_bias) stage_bias<BN>(g, s_bias[acc], n0, (warp - 2) * 32 + lane);
            tc::mbar_wait(acc_full0 + 8 * acc, (local >> 1) & 1u);
            tc::tc_fence_after();
            epi_bf16_tile<EPI, BN>(g, &tmC, tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN, m0 + q * 32, lane, n0, has_bias ? s_bias[acc] : nullptr,
                                   s_stage[warp - 2]);
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster(tc::mapa(acc_empty0 + 8 * acc, 0));   // the leader's barrier collects both CTAs
        }
        if (lane == 0) tc::tma_store_wait_all();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync();   // the peer may still be reading this CTA's shared memory (MMA) or arriving on its barriers
    if (warp == 1) tc::tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------
// TMA descriptors (driver entry point fetched at run time: the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// bf16 matrix [rows, cols] with row pitch ld (elements), tiles of box_rows x 64 columns, 128-byte swizzle
int make_map(maze_ctx* ctx, CUtensorMap* m, const void* ptr, int rows, int cols, int ld, int box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return maze_fail_arg(ctx, MAZE_E_RANGE, "cuTensorMapEncodeTiled is not available from this driver");
    if (((uintptr_t)ptr & 15) || (ld % 8) != 0) return maze_fail_arg(ctx, MAZE_E_ALIGN, "GEMM operand: 16-byte aligned base and row pitch");
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        if (ctx) snprintf(ctx->err, sizeof(ctx->err), "cuTensorMapEncodeTiled failed with %d (rows %d cols %d ld %d box %d)", (int)r, rows, cols, ld, box_rows);
        return MAZE_E_RANGE;
    }
    return 0;
}

template <int BN, int EPI, bool MN>
int launch_gemm_t(maze_ctx* ctx, const bf16* A, int lda, const bf16* B, int ldb, const GemmArgs& g, int splits, cudaStream_t st) {
    CUtensorMap ta, tb;
    if constexpr (!MN) {
        if (int rc = make_map(ctx, &ta, A, g.M, g.K, lda, BM)) return rc;
        if (int rc = make_map(ctx, &tb, B, g.N, g.K, ldb, BN)) return rc;
    } else {   // A [K, M], B [K, N]: boxes of 64 K-rows x 64 M / N elements
        if (int rc = make_map(ctx, &ta, A, g.K, g.M, lda, 64)) return rc;
        if (int rc = make_map(ctx, &tb, B, g.K, g.N, ldb, 64)) return rc;
    }
    CUtensorMap tc_out = ta;   // unused by the accumulate epilogue
    if constexpr (EPI != EPI_RED_F32) {
        if (int rc = make_map(ctx, &tc_out, g.C, g.M, g.N, g.ldc, 32)) return rc;
    }
    MAZE_CHECK(cudaFuncSetAttribute(net_gemm_kernel<BN, EPI, MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GemmCfg<BN>::SMEM));
    const int nkb = (g.K + BK - 1) / BK;
    if (splits < 1) splits = 1;
    if (splits > nkb) splits = nkb;
    GemmArgs ga = g;
    ga.splits = splits;
    const int num_tiles = ((g.M + BM - 1) / BM) * ((g.N + BN - 1) / BN) * splits;
    const int grid = num_tiles < ctx->num_sms ? num_tiles : ctx->num_sms;   // persistent: one CTA per SM walks the tiles
    net_gemm_kernel<BN, EPI, MN><<<grid, GEMM_THREADS, GemmCfg<BN>::SMEM, st>>>(ta, tb, tc_out, ga);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

template <int EPI>
int launch_gemm_pair(maze_ctx* ctx, const bf16* A, int lda, const bf16* B, int ldb, const GemmArgs& g, cudaStream_t st) {
    CUtensorMap ta, tb, tc_out;
    if (int rc = make_map(ctx, &ta, A, g.M, g.K, lda, 128)) return rc;
    if (int rc = make_map(ctx, &tb, B, g.N, g.K, ldb, 128)) return rc;
    if (int rc = make_map(ctx, &tc_out, g.C, g.M, g.N, g.ldc, 32)) return rc;
    MAZE_CHECK(cudaFuncSetAttribute(net_gemm_pair_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PAIR_SMEM));
    const int num_tiles = ((g.M + 255) / 256) * ((g.N + 255) / 256);
    int pairs = ctx->num_sms / 2;
    if (num_tiles < pairs) pairs = num_tiles;
    net_gemm_pair_kernel<EPI><<<2 * pairs, GEMM_THREADS, PAIR_SMEM, st>>>(ta, tb, tc_out, g);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

int launch_gemm(maze_ctx* ctx, int epi, int bn, const bf16* A, int lda, const bf16* B, int ldb, const GemmArgs& g, int splits, cudaStream_t st,
                bool mn_major = false) {
    if (g.M < 1 || g.N < 1 || g.K < 1 || (g.N % 8) != 0) return maze_fail_arg(ctx, MAZE_E_RANGE, "GEMM shape (N must be a multiple of 8)");
    if (epi != EPI_RED_F32 && splits > 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "split-K needs the accumulate epilogue");
    if (bn == 512) {   // CTA pairs, 256 x 256 tiles
        if (mn_major || epi == EPI_RED_F32) return maze_fail_arg(ctx, MAZE_E_RANGE, "the CTA-pair GEMM has the bf16 epilogues and K-major operands only");
        if (epi == EPI_BIAS_ACT) return launch_gemm_pair<EPI_BIAS_ACT>(ctx, A, lda, B, ldb, g, st);
        return launch_gemm_pair<EPI_MASK>(ctx, A, lda, B, ldb, g, st);
    }
    if (mn_major) {
        if (epi != EPI_RED_F32) return maze_fail_arg(ctx, MAZE_E_RANGE, "the MN-major (A^T . B) GEMM only has the accumulate epilogue");
        if ((g.M % 8) != 0) return maze_fail_arg(ctx, MAZE_E_RANGE, "MN-major GEMM: M must be a multiple of 8");
        if (bn == 256) return launch_gemm_t<256, EPI_RED_F32, true>(ctx, A, lda, B, ldb, g, splits, st);
        return launch_gemm_t<128, EPI_RED_F32, true>(ctx, A, lda, B, ldb, g, splits, st);
    }
    if (bn == 256) {
        if (epi == EPI_BIAS_ACT) return launch_gemm_t<256, EPI_BIAS_ACT, false>(ctx, A, lda, B, ldb, g, splits, st);
        if (epi == EPI_MASK) return launch_gemm_t<256, EPI_MASK, false>(ctx, A, lda, B, ldb, g, splits, st);
        return launch_gemm_t<256, EPI_RED_F32, false>(ctx, A, lda, B, ldb, g, splits, st);
    }
    if (epi == EPI_BIAS_ACT) return launch_gemm_t<128, EPI_BIAS_ACT, false>(ctx, A, lda, B, ldb, g, splits, st);
    if (epi == EPI_MASK) return launch_gemm_t<128, EPI_MASK, false>(ctx, A, lda, B, ldb, g, splits, st);
    return launch_gemm_t<128, EPI_RED_F32, false>(ctx, A, lda, B, ldb, g, splits, st);
}

// ------------------------------------------------------------------------------------------------------
// Convolution features.  Per sample, shared memory holds the image matrix
//   R[(y', x), kk]   y' = 0..33 (image row y' - 1; only y' = 1..15 are ever non-zero), x = 0..15 (column 15 is
//                    padding), kk = channel * 3 + dx' (dx' = 0..2 <-> column x + dx' - 1), 9 of 16 K slots used
// in the canonical K-major no-swizzle UMMA layout (8-row x 16-byte core matrices: the two K halves of an 8-row
// group 128 bytes apart, groups 256 bytes apart), with the 16 columns of an image row stored EVEN COLUMNS FIRST:
// row index = 16 y' + 8 (x & 1) + (x >> 1).  Then the conv outputs of one max-pool class -- the positions
// (2 py + dy_c, 2 px + dx_c) of all pooled cells (py, px) -- under vertical tap dy' are the R rows
// 16 (2 py + dy_c + dy') + 8 dx_c + px: eight consecutive rows per py, 32 rows (1 024 bytes) from one py to the
// next, i.e. ONE UMMA A operand (M = 128: py = 0..15, px = 0..7; stride-dimension offset 1 024) starting at byte
// 256 (2 (dy_c + dy') + dx_c).  Twelve MMAs per sample (4 pool classes x 3 vertical taps, N = 32 channels, K = 16)
// leave D[(py, px), 32 class + channel] in 128 TMEM columns: the four candidates of a pooled cell sit in the SAME TMEM
// lane, so the 2 x 2 max-pool is three max instructions per channel in registers -- no shuffles, and only the two
// warps that own py < 8 have an epilogue at all (the first version pooled a [position, channel] accumulator by
// exchanging values between lanes: 2 080 warp instructions of epilogue per sample against ~600 here).
// TWO samples share every MMA: sample B's image matrix starts 16 image rows (8 192 bytes) after sample A's, which is
// exactly eight py steps, so rows 0-63 of the M = 128 operand are A's pooled cells (py = 0..7) and rows 64-127 are B's.
// (The two y' rows a sample would own beyond its sixteen are only read by its dummy row py = 7.)  Warps 0-1 run A's
// epilogue from TMEM lanes 0-63, warps 2-3 run B's from lanes 64-127.
constexpr int FEAT_THREADS = 128;
constexpr int FEAT_R_ROWS = 34 * 16;               // y' = 0..15 sample A, 16..31 sample B, 32..33 zero
constexpr int FEAT_R_BYTES = FEAT_R_ROWS * 32;     // 17 408
constexpr int FEAT_W_BYTES = 3 * 32 * 32;          // three [32, 16] bf16 slices
constexpr int NET_CONV_OUT = 32 * 49;              // 1568
constexpr int NET_IN = 1600;                       // 1568 + 6, padded to a multiple of 64

__device__ __forceinline__ uint32_t r_offset(int row, int chunk) {   // byte offset of (row, K half) in the no-swizzle layout
    return (uint32_t)((row >> 3) * 256 + chunk * 128 + (row & 7) * 16);
}

// Conv2d.weight [32, 3, 3, 3] fp32 -> the three [32, 16] bf16 B operands of net_features_kernel (one per vertical tap), in the
// K-major no-swizzle core-matrix layout; run by maze_dqn_net_refresh.
__global__ void __launch_bounds__(256)
net_conv_image_kernel(const float* __restrict__ conv_w, uint8_t* __restrict__ image) {
    for (int i = threadIdx.x; i < 3 * 32 * 16; i += 256) {
        const int dy = i / 512, o = (i >> 4) & 31, kk = i & 15;
        float w = 0.f;
        if (kk < 9) w = conv_w[o * 27 + (kk / 3) * 9 + dy * 3 + (kk % 3)];
        *reinterpret_cast<bf16*>(image + dy * 1024 + r_offset(o, kk >> 3) + (kk & 7) * 2) = __float2bfloat16(w);
    }
}

// Dropout(p) between the LeakyReLU and the max-pool.  The keep mask is a pure function of (seed, draw, forward id,
// sample, element): Philox4x32-10 with key (seed lo, seed hi) and counter (element block, sample, draw lo, forward id);
// elements e = ((py * 7 + px) * 32 + channel) * 4 + 2 dy + dx of the 14 x 14 positions the pool reads, eight per block
// (16-bit draw k = e % 8 is bits 16 (k & 1) .. + 15 of word k / 2), kept iff draw < threshold.
struct NetDropout {
    uint32_t k0, k1;      // key: the dropout seed
    uint32_t draw;        // counter word 2: low 32 bits of maze_dqn_net.draw
    uint32_t fwd;         // counter word 3: 0 source on s, 1 source on s', 2 target on s', 3 maze_dqn_forward / _features
    uint32_t threshold;   // round(65536 (1 - p)): P(keep) = threshold / 65536
    float scale;          // fp32(1 / (1 - p))
};

// The 128 keep bits of one pooled cell (bit 4 channel + 2 dy + dx of keep[channel / 8]): 16 consecutive Philox blocks,
// shifted in from the top one byte per block.  Not unrolled: sixteen interleaved blocks took 246 registers, which would
// halve the kernel's four CTAs per SM.
__device__ __forceinline__ void dropout_keep_bits(const NetDropout& d, int smp, int cell, uint32_t (&keep)[4]) {
#pragma unroll 1
    for (int j = 0; j < 16; ++j) {   // block 16 cell + j: channels 2 j and 2 j + 1, four pool candidates each
        Philox ph;
        ph.k0 = d.k0;
        ph.k1 = d.k1;
        ph.c0 = (uint32_t)(16 * cell + j);
        ph.c1 = (uint32_t)smp;
        ph.c2 = d.draw;
        ph.c3 = d.fwd;
        ph.refill();
        const uint32_t o[4] = {ph.o0, ph.o1, ph.o2, ph.o3};
        uint32_t bits = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) bits |= (((o[k >> 1] >> (16 * (k & 1))) & 0xffffu) < d.threshold ? 1u : 0u) << k;
        keep[0] = (keep[0] >> 8) | (keep[1] << 24);
        keep[1] = (keep[1] >> 8) | (keep[2] << 24);
        keep[2] = (keep[2] >> 8) | (keep[3] << 24);
        keep[3] = (keep[3] >> 8) | (bits << 24);
    }
}

template <bool SAVE_IDX, bool DROPOUT>
__global__ void __launch_bounds__(FEAT_THREADS, DROPOUT ? 4 : 0)   // dropout: 128 registers, no spills, so 4 CTAs per SM still fit (0: no bound)
net_features_kernel(const float* __restrict__ vec, const uint32_t* __restrict__ win, int n, const uint4* __restrict__ conv_w_image,
                    const float* __restrict__ conv_b, bf16* __restrict__ X, uint8_t* __restrict__ pool_idx, const NetDropout drop) {
    __shared__ __align__(128) uint8_t sR[FEAT_R_BYTES];
    __shared__ __align__(128) uint8_t sW[FEAT_W_BYTES];
    __shared__ __align__(16) bf16 sfeat[2][NET_CONV_OUT];
    __shared__ __align__(16) uint8_t sidx[2][SAVE_IDX ? NET_CONV_OUT : 16];
    __shared__ float sbias[32];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        tc::mbar_init(tc::smem_u32(&bar), 1);
        tc::mbar_fence_init();
    }
    if (warp == 0) {
        tc::tmem_alloc(tc::smem_u32(&tmem_slot), 128);
        tc::tmem_relinquish();
    }
    for (int i = tid * 16; i < FEAT_R_BYTES; i += FEAT_THREADS * 16) *reinterpret_cast<uint4*>(sR + i) = make_uint4(0, 0, 0, 0);
    // weight slices sW[dy][o][kk] = conv_w[o][c][dy][dx], kk = c * 3 + dx, already in the operand layout: net_conv_image_kernel
    // builds the 3 KB image once per weight update (a CTA lives for about seven iterations: building it here from the fp32
    // weights was 12 % of this kernel's time, ncu r02t)
    for (int i = tid; i < FEAT_W_BYTES / 16; i += FEAT_THREADS) reinterpret_cast<uint4*>(sW)[i] = __ldg(conv_w_image + i);
    if (tid < 32) sbias[tid] = conv_b[tid];
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    const uint32_t bar_a = tc::smem_u32(&bar), r_base = tc::smem_u32(sR), w_base = tc::smem_u32(sW);
    uint32_t phase = 0;

    for (int s0 = 2 * blockIdx.x; s0 < n; s0 += 2 * gridDim.x) {
        // ---- build both image matrices from the packed windows (word ch * 8 + k: window rows 2 k in bits 0-14, 2 k + 1 in
        //      bits 16-30): 2 x 256 rows, four per thread
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = tid + FEAT_THREADS * k;          // 0..511: sample r >> 8, y' = (r >> 4) & 15, x = r & 15
            const int smp = s0 + (r >> 8);
            const int iy = ((r >> 4) & 15) - 1, x = r & 15;
            uint32_t v9 = 0;
            if (iy >= 0 && smp < n) {
                const uint32_t* words = win + (size_t)smp * MAZE_WINDOW_WORDS;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const uint32_t rowbits = (__ldg(words + c * 8 + (iy >> 1)) >> ((iy & 1) * 16)) & 0x7fffu;
                    v9 |= (((rowbits << 1) >> x) & 7u) << (3 * c);   // columns x - 1, x, x + 1
                }
            }
            uint32_t w[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) {   // bf16 1.0 = 0x3F80
                const uint32_t b2 = (v9 >> (2 * j)) & 3u;
                w[j] = (b2 & 1u) * 0x3F80u + (b2 >> 1) * 0x3F800000u;
            }
            const int row = (r & ~15) + ((x & 1) << 3) + (x >> 1);   // even columns first
            *reinterpret_cast<uint4*>(sR + r_offset(row, 0)) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(sR + r_offset(row, 1)) = make_uint4(w[4] & 0xffffu, 0, 0, 0);
        }
        tc::fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            constexpr uint32_t idesc = tc::idesc_bf16(128, 32);
#pragma unroll
            for (int cls = 0; cls < 4; ++cls)
#pragma unroll
                for (int dy = 0; dy < 3; ++dy) {
                    const uint64_t da = tc::smem_desc(r_base + (uint32_t)(2 * ((cls >> 1) + dy) + (cls & 1)) * 256u, 128, 1024, tc::SWIZZLE_NONE);
                    const uint64_t db = tc::smem_desc(w_base + (uint32_t)dy * 1024u, 128, 256, tc::SWIZZLE_NONE);
                    tc::umma_bf16(tmem_base + (uint32_t)cls * 32u, da, db, idesc, (uint32_t)(dy != 0));
                }
            tc::umma_commit(bar_a);
        }
        [[maybe_unused]] uint32_t keep[4] = {0u, 0u, 0u, 0u};
        if constexpr (DROPOUT) {   // the mask is drawn while the MMAs run
            const int py = (warp & 1) * 4 + (lane >> 3), px = lane & 7;
            if (s0 + (warp >> 1) < n && py < 7 && px < 7) dropout_keep_bits(drop, s0 + (warp >> 1), py * 7 + px, keep);
        }
        tc::mbar_wait(bar_a, phase);
        phase ^= 1u;
        tc::tc_fence_after();
        // ---- epilogue: warp pair (warp >> 1) owns sample s0 + (warp >> 1); its lanes are the pooled cells py = 4 (warp & 1) +
        //      lane / 8, px = lane % 8.  2 x 2 max-pool over the four class blocks (first maximum in scan order wins), bias,
        //      LeakyReLU.
        const int half = warp >> 1;
        if constexpr (DROPOUT) {
            // Dropout sits between the LeakyReLU and the pool, so every candidate is activated and masked before the
            // comparison: candidate = kept ? fp32(LeakyReLU(acc + bias) * scale) : +0 (a dropped candidate, value 0, can
            // beat negative ones).  idx bit 2: the winner's pre-activation > 0; bit 3: the winner was dropped.
            if (s0 + half < n) {
                const int py = (warp & 1) * 4 + (lane >> 3), px = lane & 7;
                float m[32];
                uint32_t v[32];
                [[maybe_unused]] uint32_t c1 = 0, c2 = 0, cpos = 0, cdrop = 0;   // bit ch: the winner's class bits, sign, dropped
#pragma unroll
                for (int cls = 0; cls < 4; ++cls) {
                    tc::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)cls * 32u, v);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int ch = 0; ch < 32; ++ch) {
                        const float x = __uint_as_float(v[ch]) + sbias[ch];
                        const bool kept = (keep[ch >> 3] >> (((ch & 7) << 2) | cls)) & 1u;
                        const float y = kept ? (x > 0.f ? x : LRELU_SLOPE * x) * drop.scale : 0.f;
                        const bool take = cls == 0 || y > m[ch];
                        m[ch] = take ? y : m[ch];
                        if constexpr (SAVE_IDX) {
                            const uint32_t bit = 1u << ch;
                            if (cls & 1) c1 = take ? (c1 | bit) : c1; else c1 = take ? (c1 & ~bit) : c1;
                            if (cls & 2) c2 = take ? (c2 | bit) : c2;
                            cpos = take ? (x > 0.f ? (cpos | bit) : (cpos & ~bit)) : cpos;
                            cdrop = take ? (kept ? (cdrop & ~bit) : (cdrop | bit)) : cdrop;
                        }
                    }
                }
                if (py < 7 && px < 7) {
                    const int q = py * 7 + px;
#pragma unroll
                    for (int ch = 0; ch < 32; ++ch) {
                        if constexpr (SAVE_IDX)
                            sidx[half][ch * 49 + q] = (uint8_t)(((c1 >> ch) & 1u) | (((c2 >> ch) & 1u) << 1) | (((cpos >> ch) & 1u) << 2) | (((cdrop >> ch) & 1u) << 3));
                        sfeat[half][ch * 49 + q] = __float2bfloat16(m[ch]);
                    }
                }
            }
        } else if (s0 + half < n) {
            const int py = (warp & 1) * 4 + (lane >> 3), px = lane & 7;
            const bool valid = py < 7 && px < 7;
            float m[32];
            uint32_t v[32];
            [[maybe_unused]] uint32_t c1 = 0, c2 = 0;   // bit ch of c1 / c2: low / high bit of the winning class
            tc::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16), v);
            tc::tmem_ld_wait();
#pragma unroll
            for (int ch = 0; ch < 32; ++ch) m[ch] = __uint_as_float(v[ch]);
#pragma unroll
            for (int cls = 1; cls < 4; ++cls) {
                tc::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)cls * 32u, v);
                tc::tmem_ld_wait();
#pragma unroll
                for (int ch = 0; ch < 32; ++ch) {
                    const float x = __uint_as_float(v[ch]);
                    if constexpr (SAVE_IDX) {
                        const bool take = x > m[ch];
                        if (cls & 1) c1 = take ? (c1 | (1u << ch)) : c1; else c1 = take ? (c1 & ~(1u << ch)) : c1;
                        if (cls & 2) c2 = take ? (c2 | (1u << ch)) : c2;
                    }
                    m[ch] = fmaxf(m[ch], x);
                }
            }
            if (valid) {
                const int q = py * 7 + px;
#pragma unroll
                for (int ch = 0; ch < 32; ++ch) {
                    float x = m[ch] + sbias[ch];
                    if constexpr (SAVE_IDX) sidx[half][ch * 49 + q] = (uint8_t)(((c1 >> ch) & 1u) | (((c2 >> ch) & 1u) << 1) | (x > 0.f ? 4u : 0u));
                    x = x > 0.f ? x : LRELU_SLOPE * x;
                    sfeat[half][ch * 49 + q] = __float2bfloat16(x);
                }
            }
        }
        tc::tc_fence_before();
        __syncthreads();
        // ---- write the feature rows: 1568 conv features, 6 state floats, zero padding up to 1600
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int smp = s0 + h;
            if (smp >= n) break;
            bf16* xrow = X + (size_t)smp * NET_IN;
            for (int i = tid; i < NET_CONV_OUT / 8; i += FEAT_THREADS)
                reinterpret_cast<uint4*>(xrow)[i] = reinterpret_cast<const uint4*>(sfeat[h])[i];
            if (tid < 32) xrow[NET_CONV_OUT + tid] = __float2bfloat16(tid < 6 ? __ldg(vec + (size_t)smp * 6 + tid) : 0.f);
            if constexpr (SAVE_IDX) {
                uint8_t* irow = pool_idx + (size_t)smp * NET_CONV_OUT;
                for (int i = tid; i < NET_CONV_OUT / 16; i += FEAT_THREADS)
                    reinterpret_cast<uint4*>(irow)[i] = reinterpret_cast<const uint4*>(sidx[h])[i];
            }
        }
        // the next iteration rewrites sfeat / sidx only after its own __syncthreads
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem_base, 128);
}

// ------------------------------------------------------------------------------------------------------
// fc3 head (512 -> 4, fp32 weights, CUDA cores).  q[n, 4] for action selection.
constexpr int HEAD_THREADS = 256;
constexpr int NET_H2 = 512, NET_H1 = 1024;
constexpr size_t HEAD_LOSS_SMEM = (size_t)(2 + HEAD_THREADS / 32) * 4 * NET_H2 * sizeof(float);   // fc3 weights of both nets + one gradient copy per warp: 80 KB

// A warp owns one sample; lane l holds the 16 columns  k * 128 + 4 l + j  (k, j = 0..3) of its 512-wide rows: global
// loads are 8 bytes per lane and 256 contiguous bytes per warp, shared-memory weight reads are float4 at a 16-byte lane
// stride (conflict-free; the first version's 16 consecutive columns per lane made every weight read a 16-way bank
// conflict: ncu profiles r02n, 4.6 M conflicts, short-scoreboard stalls).
__device__ __forceinline__ int head_col(int lane, int i) { return (i >> 2) * 128 + lane * 4 + (i & 3); }

__device__ __forceinline__ void head_load16(const bf16* row, int lane, float (&h)[16]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint2 w = __ldg(reinterpret_cast<const uint2*>(row + k * 128 + lane * 4));
        h[4 * k + 0] = __uint_as_float(w.x << 16);
        h[4 * k + 1] = __uint_as_float(w.x & 0xffff0000u);
        h[4 * k + 2] = __uint_as_float(w.y << 16);
        h[4 * k + 3] = __uint_as_float(w.y & 0xffff0000u);
    }
}

// The same row as raw words (prefetch one sample ahead), and their expansion
__device__ __forceinline__ void head_load_raw(const bf16* row, int lane, uint2 (&w)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = __ldg(reinterpret_cast<const uint2*>(row + k * 128 + lane * 4));
}
__device__ __forceinline__ void head_expand(const uint2 (&w)[4], float (&h)[16]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        h[4 * k + 0] = __uint_as_float(w[k].x << 16);
        h[4 * k + 1] = __uint_as_float(w[k].x & 0xffff0000u);
        h[4 * k + 2] = __uint_as_float(w[k].y << 16);
        h[4 * k + 3] = __uint_as_float(w[k].y & 0xffff0000u);
    }
}

__device__ __forceinline__ float head_dot(const float (&h)[16], const float* w_row, int lane) {   // w_row: 512 floats in shared memory
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float4 w = *reinterpret_cast<const float4*>(w_row + k * 128 + lane * 4);
        acc = fmaf(h[4 * k + 0], w.x, acc);
        acc = fmaf(h[4 * k + 1], w.y, acc);
        acc = fmaf(h[4 * k + 2], w.z, acc);
        acc = fmaf(h[4 * k + 3], w.w, acc);
    }
    return acc;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(HEAD_THREADS)
net_head_q_kernel(const bf16* __restrict__ h2, int n, const float* __restrict__ w3, const float* __restrict__ b3, float* __restrict__ q) {
    __shared__ __align__(16) float sw[4 * NET_H2];
    for (int i = threadIdx.x; i < 4 * NET_H2; i += HEAD_THREADS) sw[i] = w3[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int s = blockIdx.x * (HEAD_THREADS / 32) + (threadIdx.x >> 5); s < n; s += gridDim.x * (HEAD_THREADS / 32)) {
        float h[16];
        head_load16(h2 + (size_t)s * NET_H2, lane, h);
        float acc[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) acc[a] = warp_sum(head_dot(h, sw + a * NET_H2, lane));
        if (lane < 4) q[(size_t)s * 4 + lane] = (lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3]) + b3[lane];
    }
}

// Loss and the gradient at the head (ddqn_agent.py:131-143): q(s, a) from the source net, a* = argmax_a' q_source(s', a'),
// y = r + gamma * q_target(s', a*), loss = mean (q(s, a) - y)^2.  Writes dL/d(pre-ReLU h2) [n, 512] bf16 and accumulates the
// fc3 gradients.  UPDATE == UPDATE_MAX_TARGET: the DQN target y = r + gamma * max_a' q_target(s', a') (no source forward on
// s': h2_sn is not read and may be null).
enum { UPDATE_DOUBLE_Q = 0, UPDATE_MAX_TARGET = 1 };
template <int UPDATE>
__global__ void __launch_bounds__(HEAD_THREADS, 2)
net_head_loss_kernel(const bf16* __restrict__ h2_s, const bf16* __restrict__ h2_sn, const bf16* __restrict__ h2_tn, int n,
                     const float* __restrict__ w3, const float* __restrict__ b3, const float* __restrict__ tw3, const float* __restrict__ tb3,
                     const uint8_t* __restrict__ action, const float* __restrict__ reward, float gamma, bf16* __restrict__ dh2,
                     float* __restrict__ gw3, float* __restrict__ gb3, float* __restrict__ loss, float* __restrict__ qsa_out) {
    // dynamic shared memory: fc3 weights of both nets (2 x 8 KB) and ONE d fc3.weight accumulator PER WARP (8 x 8 KB), in
    // lane-major order (entry (a, i, lane) <-> column head_col(lane, i)).  A warp's lanes own distinct entries of its copy, so
    // the per-sample update is a plain conflict-free read-add-write: the single shared copy it replaces needed a shared
    // float atomic per entry -- a CAS loop, 21 % of this kernel's stall samples (ncu profiles/r02zz_head_details.txt).
    extern __shared__ __align__(16) float head_smem[];
    float* const sw = head_smem;
    float* const stw = sw + 4 * NET_H2;
    float* const sgw_all = stw + 4 * NET_H2;
    __shared__ float sgb[4], sloss;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* const sgw = sgw_all + warp * (4 * NET_H2);
    // the first sample's rows are requested before the weights: the two round trips to memory overlap
    const int stride = gridDim.x * (HEAD_THREADS / 32);
    int s = blockIdx.x * (HEAD_THREADS / 32) + warp;
    uint2 ra[4], rb[4], rc[4];
    int act_next = 0;
    float rew_next = 0.f;
    if (s < n) {
        head_load_raw(h2_s + (size_t)s * NET_H2, lane, ra);
        if constexpr (UPDATE == UPDATE_DOUBLE_Q) head_load_raw(h2_sn + (size_t)s * NET_H2, lane, rb);
        head_load_raw(h2_tn + (size_t)s * NET_H2, lane, rc);
        act_next = action[s] & 3;
        rew_next = reward[s];
    }
    for (int i = threadIdx.x; i < NET_H2; i += HEAD_THREADS) {   // 4 x 512 floats each, 16 bytes per load
        reinterpret_cast<float4*>(sw)[i] = __ldg(reinterpret_cast<const float4*>(w3) + i);
        reinterpret_cast<float4*>(stw)[i] = __ldg(reinterpret_cast<const float4*>(tw3) + i);
    }
    for (int i = threadIdx.x; i < (HEAD_THREADS / 32) * NET_H2; i += HEAD_THREADS) reinterpret_cast<float4*>(sgw_all)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (threadIdx.x < 4) sgb[threadIdx.x] = 0.f;
    if (threadIdx.x == 0) sloss = 0.f;
    __syncthreads();
    const float inv_n = 1.f / (float)n;
    float gb_acc = 0.f, loss_acc = 0.f;   // lane a < 4 collects d fc3.bias[a]; lane 0 the loss
    // The loop is a chain of global loads -> dot products -> butterfly sums with two CTAs of eight warps per SM: the next
    // sample's three rows are fetched while the current one is reduced (ncu r02t: 82 % of the cycles had no eligible warp).
    for (; s < n; s += stride) {
        float h[16], hn[16], ht[16];
        head_expand(ra, h);
        if constexpr (UPDATE == UPDATE_DOUBLE_Q) head_expand(rb, hn);
        head_expand(rc, ht);
        const int act = act_next;
        const float rew = rew_next;
        if (s + stride < n) {
            const size_t t = (size_t)(s + stride);
            head_load_raw(h2_s + t * NET_H2, lane, ra);
            if constexpr (UPDATE == UPDATE_DOUBLE_Q) head_load_raw(h2_sn + t * NET_H2, lane, rb);
            head_load_raw(h2_tn + t * NET_H2, lane, rc);
            act_next = action[t] & 3;
            rew_next = reward[t];
        }
        float qs[4], qn[4], qt[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            qs[a] = head_dot(h, sw + a * NET_H2, lane);
            if constexpr (UPDATE == UPDATE_DOUBLE_Q) qn[a] = head_dot(hn, sw + a * NET_H2, lane);
            qt[a] = head_dot(ht, stw + a * NET_H2, lane);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) {   // twelve independent butterfly reductions, interleaved by the compiler
            qs[a] = warp_sum(qs[a]) + b3[a];
            if constexpr (UPDATE == UPDATE_DOUBLE_Q) qn[a] = warp_sum(qn[a]) + b3[a];
            qt[a] = warp_sum(qt[a]) + tb3[a];
        }
        int best = 0;   // .max(1)[1]: first maximum
        if constexpr (UPDATE == UPDATE_DOUBLE_Q) {
#pragma unroll
            for (int a = 1; a < 4; ++a)
                if (qn[a] > qn[best]) best = a;
        }
        const float qsa = act == 0 ? qs[0] : act == 1 ? qs[1] : act == 2 ? qs[2] : qs[3];
        const float qtb = UPDATE == UPDATE_MAX_TARGET ? fmaxf(fmaxf(qt[0], qt[1]), fmaxf(qt[2], qt[3]))   // .max(1)[0]
                                                      : best == 0 ? qt[0] : best == 1 ? qt[1] : best == 2 ? qt[2] : qt[3];
        const float target = qtb * gamma + rew;
        const float d = qsa - target;
        const float gq = 2.f * d * inv_n;   // d mean((q - y)^2) / d q
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float4 w = *reinterpret_cast<const float4*>(sw + act * NET_H2 + k * 128 + lane * 4);
            uint2 out;   // ReLU'
            out.x = tc::pack_bf16x2(h[4 * k + 0] > 0.f ? gq * w.x : 0.f, h[4 * k + 1] > 0.f ? gq * w.y : 0.f);
            out.y = tc::pack_bf16x2(h[4 * k + 2] > 0.f ? gq * w.z : 0.f, h[4 * k + 3] > 0.f ? gq * w.w : 0.f);
            *reinterpret_cast<uint2*>(dh2 + (size_t)s * NET_H2 + k * 128 + lane * 4) = out;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) sgw[act * NET_H2 + i * 32 + lane] += gq * h[i];   // this warp's copy, this lane's entries
        if (lane == act) gb_acc += gq;
        if (lane == 0) {
            loss_acc += d * d * inv_n;
            if (qsa_out) qsa_out[s] = qsa;
        }
    }
    if (lane < 4 && gb_acc != 0.f) atomicAdd(&sgb[lane], gb_acc);
    if (lane == 0) atomicAdd(&sloss, loss_acc);
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * NET_H2; i += HEAD_THREADS) {
        float v = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < HEAD_THREADS / 32; ++w8) v += sgw_all[w8 * (4 * NET_H2) + i];
        if (v != 0.f) atomicAdd(gw3 + (i >> 9) * NET_H2 + head_col(i & 31, (i >> 5) & 15), v);
    }
    if (threadIdx.x < 4) atomicAdd(gb3 + threadIdx.x, sgb[threadIdx.x]);
    if (threadIdx.x == 0) atomicAdd(loss, sloss);
}

// ------------------------------------------------------------------------------------------------------
// out[c] += sum_r in[r, c]: the bias gradients (column sums of dL/d pre-activation).  One CTA per 256 columns x 64 rows:
// a warp reads 512 contiguous bytes of a row (16 bytes per lane) and keeps its eight row loads in flight together -- the
// first version walked 64 rows per warp one 4-byte load at a time (12 us for 8 MB: a latency chain, not bandwidth).
constexpr int COLSUM_COLS = 256, COLSUM_ROWS = 64;
__global__ void __launch_bounds__(256)
net_colsum_kernel(const bf16* __restrict__ in, int R, int C, int ld, float* __restrict__ out) {
    __shared__ float part[8][COLSUM_COLS];
    const int c0 = blockIdx.x * COLSUM_COLS, r0 = blockIdx.y * COLSUM_ROWS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = c0 + 8 * lane;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c + 8 <= C) {
        uint4 v[COLSUM_ROWS / 8];
#pragma unroll
        for (int i = 0; i < COLSUM_ROWS / 8; ++i) {
            const int r = r0 + warp + 8 * i;
            v[i] = r < R ? __ldg(reinterpret_cast<const uint4*>(in + (size_t)r * ld + c)) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int i = 0; i < COLSUM_ROWS / 8; ++i) {
            const uint32_t w[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                acc[2 * u] += __uint_as_float(w[u] << 16);
                acc[2 * u + 1] += __uint_as_float(w[u] & 0xffff0000u);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) part[warp][8 * lane + u] = acc[u];
    __syncthreads();
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) v += part[k][threadIdx.x];
    if (c0 + (int)threadIdx.x < C && v != 0.f) atomicAdd(out + c0 + threadIdx.x, v);
}

// ------------------------------------------------------------------------------------------------------
// Convolution weight / bias gradient from dL/dX (conv part), the saved pool choices and the packed windows, on the
// tensor cores.  Per sample
//   D[o, kk] += sum_p A[o, p] * B[kk, p],   p = y * 16 + x over the 16 x 16 padded window positions (K = 256)
//   A[o, p]  = dL/d(conv output o at p): the pooled gradient dX[o, q] * LeakyReLU', routed to its max-pool winner
//   B[kk, p] = window bit of tap kk = c * 9 + dy * 3 + dx at p (the window shifted by (dy - 1, dx - 1));
//              kk = 27 is all ones, so column 27 of D is the bias gradient; kk = 28 .. 31 stay zero
// Both operands are K-major without swizzle (8 consecutive positions = one 16-byte core-matrix row, the core
// matrices of one 8-position group 128 bytes apart along M / N, the groups 64 (32) x 16 bytes apart along K);
// UMMA M = 64 (rows 32 .. 63 of A stay zero), N = 32, 14 MMAs of K = 16 per sample (one per window row).  One
// operand buffer per CTA (48 KB) and four CTAs per SM: while one CTA waits for its MMAs the others build.  The
// accumulator stays in TMEM over all the samples of a CTA and is added to the global gradient once (M = 64: row r
// lives in TMEM lane 32 (r / 16) + r % 16).
constexpr int CB_THREADS = 256;
constexpr uint32_t CB_A_BYTES = 64 * 256 * 2, CB_B_BYTES = 32 * 256 * 2;
constexpr size_t CB_SMEM = CB_A_BYTES + CB_B_BYTES + 128;   // 48 KB (+ 9 KB static staging): three CTAs per SM overlap each other's build / MMA phases
constexpr int CB_B_UNITS = 27 * 28;                          // (tap, window row 0..13, half row)

// DROPOUT: the pool winner's gradient passes the Dropout backward first (0 if idx bit 3 says it was dropped, else times
// drop_scale), then the LeakyReLU backward -- autograd's order.
template <bool DROPOUT>
__global__ void __launch_bounds__(CB_THREADS, 3)
net_conv_bwd_tc_kernel(const bf16* __restrict__ dX, const uint8_t* __restrict__ pool_idx, const uint32_t* __restrict__ win, int n,
                       float* __restrict__ gconv_w, float* __restrict__ gconv_b, float drop_scale) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    // One sample's gradient row (1 568 bf16) and pool choices (1 568 bytes), double-buffered: fetched from global memory
    // with coalesced 16-byte loads one sample ahead.  Reading them straight from global with this kernel's (channel,
    // pooled position) thread mapping made every 1- and 2-byte load touch 32 sectors -- L1 tag look-ups, not bytes,
    // bounded the first version (87 us per 8 192 samples, profiles/r02m_net_launches_summary.txt).
    __shared__ __align__(16) bf16 s_g[2][NET_CONV_OUT];
    __shared__ __align__(16) uint8_t s_i[2][NET_CONV_OUT];
    __shared__ uint32_t s_w[2][MAZE_WINDOW_WORDS];   // and its packed window
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t* const A = smem_raw + ((128u - (tc::smem_u32(smem_raw) & 127u)) & 127u);
    uint8_t* const B = A + CB_A_BYTES;
    for (uint32_t i = tid * 16; i < CB_A_BYTES + CB_B_BYTES; i += CB_THREADS * 16) *reinterpret_cast<uint4*>(A + i) = make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        tc::mbar_init(tc::smem_u32(&bar), 1);
        tc::mbar_fence_init();
    }
    if (warp == 0) {
        tc::tmem_alloc(tc::smem_u32(&tmem_slot), 32);
        tc::tmem_relinquish();
    }
    __syncthreads();
    if (tid < 32)   // the all-ones row kk = 27 of B: 32 position groups
        *reinterpret_cast<uint4*>(B + tid * 512 + (27 >> 3) * 128 + (27 & 7) * 16) = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    const uint32_t bar_a = tc::smem_u32(&bar);
    // A units of this thread: channel o, pooled row py, half h (14 units per channel over 8 thread groups)
    const int o = tid & 31, part = tid >> 5;
    const uint32_t a_row = (uint32_t)((o >> 3) * 128 + (o & 7) * 16);
    // B units of this thread (fixed over the samples): tap kk, window row y, half h
    int b_word[3], b_shift[3], b_sh8[3];
    uint32_t b_off[3];
    bool b_on[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int u = tid + CB_THREADS * j;
        const int kk = u % 27, yh = u / 27;
        const int y = yh >> 1, h = yh & 1, c = kk / 9, dy = (kk % 9) / 3, dx = kk % 3, iy = y + dy - 1;
        b_on[j] = u < CB_B_UNITS && iy >= 0 && iy < MAZE_WINDOW;
        b_word[j] = c * 8 + (max(iy, 0) >> 1);
        b_shift[j] = (iy & 1) * 16;
        b_sh8[j] = 8 * h + dx;
        b_off[j] = u < CB_B_UNITS ? (uint32_t)yh * 512u + (uint32_t)((kk >> 3) * 128 + (kk & 7) * 16) : 0xffffffffu;
    }
    auto fetch = [&](int smp, uint4& gq, uint4& iq, uint32_t& wq) {   // this thread's share of the sample's gradient row / pool choices / window
        gq = iq = make_uint4(0, 0, 0, 0);
        wq = 0;
        if (smp < n) {
            if (tid < NET_CONV_OUT / 8) gq = __ldg(reinterpret_cast<const uint4*>(dX + (size_t)smp * NET_IN) + tid);
            if (tid < NET_CONV_OUT / 16) iq = __ldg(reinterpret_cast<const uint4*>(pool_idx + (size_t)smp * NET_CONV_OUT) + tid);
            if (tid >= 224 && tid < 224 + MAZE_WINDOW_WORDS) wq = __ldg(win + (size_t)smp * MAZE_WINDOW_WORDS + (tid - 224));
        }
    };
    auto stash = [&](int buf, const uint4& gq, const uint4& iq, uint32_t wq) {
        if (tid < NET_CONV_OUT / 8) reinterpret_cast<uint4*>(s_g[buf])[tid] = gq;
        if (tid < NET_CONV_OUT / 16) reinterpret_cast<uint4*>(s_i[buf])[tid] = iq;
        if (tid >= 224 && tid < 224 + MAZE_WINDOW_WORDS) s_w[buf][tid - 224] = wq;
    };
    {
        uint4 gq, iq;
        uint32_t wq;
        fetch(blockIdx.x, gq, iq, wq);
        stash(0, gq, iq, wq);
    }
    __syncthreads();
    uint32_t it = 0;
    for (int s = blockIdx.x; s < n; s += gridDim.x, ++it) {
        const int buf = (int)(it & 1u);
        uint4 next_g, next_i;
        uint32_t next_w;
        fetch(s + (int)gridDim.x, next_g, next_i, next_w);   // in flight while this sample is built
        // everything that does not touch the operand buffers (the previous sample's MMAs may still be reading them) first
        uint32_t bits8[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            bits8[j] = 0;
            if (b_on[j]) bits8[j] = (((((s_w[buf][b_word[j]] >> b_shift[j]) & 0x7fffu) << 1) >> b_sh8[j])) & 0xffu;
        }
        uint32_t top[2][4], bot[2][4];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int u = part + 8 * k;
            const int py = u >> 1, h = u & 1;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t word = 0, b = 0;
                if (u < 14 && 4 * h + j < 7) {
                    const int at = o * 49 + py * 7 + 4 * h + j;
                    b = s_i[buf][at];
                    float gv = __bfloat162float(s_g[buf][at]);
                    if constexpr (DROPOUT) gv = (b & 8u) ? 0.f : gv * drop_scale;
                    if (!(b & 4u)) gv *= LRELU_SLOPE;
                    const uint32_t hb = (uint32_t)__bfloat16_as_ushort(__float2bfloat16(gv));
                    word = (b & 1u) ? hb << 16 : hb;       // columns 2 px and 2 px + 1 share a word
                }
                top[k][j] = (b & 2u) ? 0u : word;
                bot[k][j] = (b & 2u) ? word : 0u;
            }
        }
        if (it >= 1) tc::mbar_wait(bar_a, (it - 1u) & 1u);   // the previous sample's MMAs have read A and B
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int u = part + 8 * k;
            if (u < 14) {
                const int py = u >> 1, h = u & 1;
                *reinterpret_cast<uint4*>(A + (uint32_t)(4 * py + h) * 1024u + a_row) = make_uint4(top[k][0], top[k][1], top[k][2], top[k][3]);
                *reinterpret_cast<uint4*>(A + (uint32_t)(4 * py + 2 + h) * 1024u + a_row) = make_uint4(bot[k][0], bot[k][1], bot[k][2], bot[k][3]);
            }
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (b_off[j] != 0xffffffffu) {
                uint32_t w[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t b2 = (bits8[j] >> (2 * q)) & 3u;
                    w[q] = (b2 & 1u) * 0x3F80u + (b2 >> 1) * 0x3F800000u;
                }
                *reinterpret_cast<uint4*>(B + b_off[j]) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
        stash(buf ^ 1, next_g, next_i, next_w);   // the other stage: its last readers passed the barrier of the previous iteration
        tc::fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            constexpr uint32_t idesc = tc::idesc_bf16(64, 32);
            const uint32_t a_addr = tc::smem_u32(A), b_addr = tc::smem_u32(B);
#pragma unroll
            for (int j = 0; j < 14; ++j)   // positions 16 j .. 16 j + 15 = window row j (rows 14, 15 contribute nothing)
                tc::umma_bf16(tmem_base, tc::smem_desc(a_addr + j * 2048u, 1024, 128, tc::SWIZZLE_NONE),
                              tc::smem_desc(b_addr + j * 1024u, 512, 128, tc::SWIZZLE_NONE), idesc, (uint32_t)((it | (uint32_t)j) != 0));
            tc::umma_commit(bar_a);
        }
    }
    if (it > 0) {
        tc::mbar_wait(bar_a, (it - 1u) & 1u);
        tc::tc_fence_after();
        if (warp < 2) {
            uint32_t v[32];
            tc::tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16), v);
            tc::tmem_ld_wait();
            if (lane < 16) {
                const int ch = warp * 16 + lane;
#pragma unroll
                for (int kk = 0; kk < 27; ++kk) atomicAdd(gconv_w + ch * 27 + kk, __uint_as_float(v[kk]));
                atomicAdd(gconv_b + ch, __uint_as_float(v[27]));
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem_base, 32);
}

// ------------------------------------------------------------------------------------------------------
// AdamW (torch.optim.AdamW defaults, ddqn_agent.py:91) with the reference's elementwise gradient clamp
// (ddqn_agent.py:146-147).  Zeroes the gradient accumulators for the next step.
__global__ void __launch_bounds__(256)
net_adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int count, float lr, float beta1,
                 float beta2, float eps, float wd, float bc1, float bc2_sqrt, float grad_scale, float clamp) {
    const int i = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (i >= count) return;
    float4 P = *reinterpret_cast<float4*>(p + i), G = *reinterpret_cast<float4*>(g + i), M = *reinterpret_cast<float4*>(m + i),
           V = *reinterpret_cast<float4*>(v + i);
    float* pp = &P.x;
    float* gg = &G.x;
    float* mm = &M.x;
    float* vv = &V.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float gr = gg[k] * grad_scale;
        if (clamp > 0.f) gr = fminf(fmaxf(gr, -clamp), clamp);
        pp[k] *= 1.f - lr * wd;
        mm[k] = beta1 * mm[k] + (1.f - beta1) * gr;
        vv[k] = beta2 * vv[k] + (1.f - beta2) * gr * gr;
        const float denom = sqrtf(vv[k]) / bc2_sqrt + eps;
        pp[k] -= (lr / bc1) * (mm[k] / denom);
    }
    *reinterpret_cast<float4*>(p + i) = P;
    *reinterpret_cast<float4*>(m + i) = M;
    *reinterpret_cast<float4*>(v + i) = V;
    *reinterpret_cast<float4*>(g + i) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// fp32 [R, C] master weights -> bf16 [R, C] (GEMM B operand of the forward pass) and optionally bf16 [C, R]
// (B operand of the backward-data pass)
__global__ void __launch_bounds__(256)
net_refresh_kernel(const float* __restrict__ w, int R, int C, bf16* __restrict__ wb, bf16* __restrict__ wt) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        const float x = (r < R && c < C) ? w[(size_t)r * C + c] : 0.f;
        tile[i][tx] = x;
        if (r < R && c < C) wb[(size_t)r * C + c] = __float2bfloat16(x);
    }
    if (!wt) return;
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (r < R && c < C) wt[(size_t)c * R + r] = __float2bfloat16(tile[tx][i]);
    }
}

// memory.sample(n) that leaves the windows bit-packed (the network kernels read them as they are)
__global__ void __launch_bounds__(256)
net_sample_packed_kernel(maze_replay r, int n, unsigned long long seed, unsigned long long draw, float* __restrict__ vec,
                         uint32_t* __restrict__ win, float* __restrict__ next_vec, uint32_t* __restrict__ next_win,
                         uint8_t* __restrict__ action, float* __restrict__ reward) {
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (k >= n) return;
    const unsigned long long pushed = *r.pushed;
    const unsigned long long filled = pushed < (unsigned long long)r.capacity ? pushed : (unsigned long long)r.capacity;
    if (filled == 0) return;
    const size_t slot = replay_slot(r, filled, n, seed, draw, k);   // the same draw as maze_dqn_sample
    if (lane < 6) {
        vec[(size_t)k * 6 + lane] = r.vec[slot * 6 + lane];
        next_vec[(size_t)k * 6 + lane] = r.next_vec[slot * 6 + lane];
    }
    if (lane < MAZE_WINDOW_WORDS) {
        win[(size_t)k * MAZE_WINDOW_WORDS + lane] = r.win[slot * MAZE_WINDOW_WORDS + lane];
        next_win[(size_t)k * MAZE_WINDOW_WORDS + lane] = r.next_win[slot * MAZE_WINDOW_WORDS + lane];
    }
    if (lane == 0) {
        action[k] = r.action[slot];
        reward[k] = r.reward[slot];
    }
}

// ------------------------------------------------------------------------------------------------------
// Workspace carving (bf16 activations; rows padded to a multiple of 128 so every TMA box starts in bounds)
struct Workspace {
    int n, np;   // batch, padded batch
    bf16 *X, *h1, *h1t_tn, *h2, *h2_tn, *dh2, *dh1, *dX;
    uint8_t* idx;
    uint8_t* conv_image[2];   // source / target net: conv weights as UMMA operands (net_conv_image_kernel)
    float* q;
    size_t bytes;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

Workspace carve(void* base, int n) {
    Workspace w{};
    w.n = n;
    w.np = (n + 127) / 128 * 128;
    const size_t np = (size_t)w.np;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* p = base ? static_cast<uint8_t*>(base) + off : nullptr;
        off += align256(bytes);
        return p;
    };
    w.X = (bf16*)take(2 * np * NET_IN * 2);          // rows 0..np-1 state, np..2np-1 next state
    w.h1 = (bf16*)take(2 * np * NET_H1 * 2);         // source net on both halves
    w.h1t_tn = (bf16*)take(np * NET_H1 * 2);         // target net on the next states
    w.h2 = (bf16*)take(2 * np * NET_H2 * 2);
    w.h2_tn = (bf16*)take(np * NET_H2 * 2);
    w.dh2 = (bf16*)take(np * NET_H2 * 2);
    w.dh1 = (bf16*)take(np * NET_H1 * 2);
    w.dX = (bf16*)take(np * NET_IN * 2);
    w.idx = (uint8_t*)take(np * NET_CONV_OUT);
    w.q = (float*)take(2 * np * 4 * sizeof(float));
    w.conv_image[0] = (uint8_t*)take(FEAT_W_BYTES);
    w.conv_image[1] = (uint8_t*)take(FEAT_W_BYTES);
    w.bytes = off;
    return w;
}

int check_net(maze_ctx* ctx, const maze_dqn_net* net, bool train) {
    if (!net) return maze_fail_arg(ctx, MAZE_E_NULL, "net");
    if (!net->params || !net->target || !net->w1_bf16 || !net->w2_bf16 || !net->tw1_bf16 || !net->tw2_bf16 || !net->workspace)
        return maze_fail_arg(ctx, MAZE_E_NULL, "net pointer");
    if (train && (!net->grads || !net->adam_m || !net->adam_v || !net->w1t_bf16 || !net->w2t_bf16 || !net->loss))
        return maze_fail_arg(ctx, MAZE_E_NULL, "net training pointer");
    if (((uintptr_t)net->params & 15) || ((uintptr_t)net->target & 15) || ((uintptr_t)net->workspace & 255))
        return maze_fail_arg(ctx, MAZE_E_ALIGN, "net params (16 bytes) / workspace (256 bytes)");
    if (!(net->dropout >= 0.f && net->dropout < 1.f)) return maze_fail_arg(ctx, MAZE_E_RANGE, "net dropout (0 <= p < 1)");
    if (net->update != 0 && net->update != 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "net update (0 double-Q, 1 max target)");
    if (net->eval != 0 && net->eval != 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "net eval (0 training, 1 evaluation)");
    return 0;
}

// The Dropout of forward `fwd`, or null when the net has none (p = 0, or evaluation mode)
const NetDropout* dropout_of(const maze_dqn_net* net, uint32_t fwd, NetDropout& d) {
    if (!(net->dropout > 0.f) || net->eval) return nullptr;
    const double keep = 1.0 - (double)net->dropout;
    d.k0 = (uint32_t)net->dropout_seed;
    d.k1 = (uint32_t)(net->dropout_seed >> 32);
    d.draw = (uint32_t)net->draw;
    d.fwd = fwd;
    d.threshold = (uint32_t)floor(65536.0 * keep + 0.5);
    d.scale = (float)(1.0 / keep);
    return &d;
}

// Split-K factor of a weight-gradient GEMM (tiles x k-blocks, persistent over `sms` CTAs): the one that minimises
// waves x (k-blocks per split + a fixed per-tile cost of about six k-blocks: pipeline fill, accumulator drain, atomics).
// fc1 at n = 8192: 56 tiles x 128 k-blocks -> 5 splits (280 tiles, 1.9 waves) instead of 4 (224 tiles, 1.5 waves run as 2).
int auto_splits(int base_tiles, int nkb, int sms) {
    int best = 1;
    float best_cost = 1e30f;
    for (int s = 1; s <= 16 && nkb / s >= 8; ++s) {
        const int waves = (base_tiles * s + sms - 1) / sms;
        const float cost = (float)waves * ((float)nkb / (float)s + 6.f);
        if (cost < best_cost * 0.98f) {   // a larger split has to pay for its extra atomics
            best_cost = cost;
            best = s;
        }
    }
    return best;
}

// In-situ kernel times: while enabled (maze_dqn_net_profile), maze_dqn_backward records a CUDA event on its stream after
// every launch; maze_dqn_net_profile_read turns the last call's events into per-launch durations.  These are the times
// the kernels take INSIDE the train step (warm L2, real clocks), which ncu's serialised cold-cache replays do not show.
struct NetProfile {
    static constexpr int CAP = 96;
    bool on = false;
    int count = 0;
    cudaEvent_t ev[CAP] = {};
    const char* label[CAP] = {};
};

inline void prof_reset(maze_ctx* ctx, cudaStream_t st) {
    NetProfile* pr = static_cast<NetProfile*>(ctx->net_profile);
    if (!pr || !pr->on) return;
    pr->count = 0;
    if (!pr->ev[0]) for (auto& e : pr->ev) cudaEventCreate(&e);
    pr->label[0] = "begin";
    cudaEventRecord(pr->ev[0], st);
    pr->count = 1;
}

inline void prof_mark(maze_ctx* ctx, cudaStream_t st, const char* label) {
    NetProfile* pr = static_cast<NetProfile*>(ctx->net_profile);
    if (!pr || !pr->on || pr->count == 0 || pr->count >= NetProfile::CAP) return;
    pr->label[pr->count] = label;
    cudaEventRecord(pr->ev[pr->count++], st);
}

int features(maze_ctx* ctx, bool save_idx, const float* vec, const uint32_t* win, int n, const float* params, const uint8_t* conv_image, bf16* X,
             uint8_t* idx, cudaStream_t st, const NetDropout* drop = nullptr) {
    const int pairs = (n + 1) / 2;   // two samples per iteration
    const int grid = pairs < ctx->num_sms * 4 ? pairs : ctx->num_sms * 4;   // 128 TMEM columns per CTA: four CTAs per SM
    const auto kernel = drop ? (save_idx ? net_features_kernel<true, true> : net_features_kernel<false, true>)
                             : (save_idx ? net_features_kernel<true, false> : net_features_kernel<false, false>);
    kernel<<<grid, FEAT_THREADS, 0, st>>>(vec, win, n, reinterpret_cast<const uint4*>(conv_image), params + MAZE_NET_OFF_CONV_B, X, idx,
                                          drop ? *drop : NetDropout{});
    MAZE_CHECK(cudaGetLastError());
    prof_mark(ctx, st, drop ? (save_idx ? "features (conv + dropout + pool, saves argmax)" : "features (conv + dropout + pool)")
                            : (save_idx ? "features (conv + pool, saves argmax)" : "features (conv + pool)"));
    return 0;
}

// Tile choice of the four K-major GEMMs of the net: CTA pairs (256 x 256) once there are at least two row blocks.
int fc_tile(int rows) { return rows > 128 ? 512 : 256; }

// X [rows, 1600] -> h1 [rows, 1024] -> h2 [rows, 512] with one net's weights
int mlp_forward(maze_ctx* ctx, const bf16* X, int rows, const bf16* w1b, const bf16* w2b, const float* params, bf16* h1, bf16* h2, cudaStream_t st) {
    GemmArgs g{};
    g.M = rows; g.N = NET_H1; g.K = NET_IN; g.C = h1; g.ldc = NET_H1; g.bias = params + MAZE_NET_OFF_B1; g.act = ACT_LRELU;
    if (int rc = launch_gemm(ctx, EPI_BIAS_ACT, fc_tile(rows), X, NET_IN, w1b, NET_IN, g, 1, st)) return rc;
    prof_mark(ctx, st, "fc1 forward GEMM");
    g = GemmArgs{};
    g.M = rows; g.N = NET_H2; g.K = NET_H1; g.C = h2; g.ldc = NET_H2; g.bias = params + MAZE_NET_OFF_B2; g.act = ACT_RELU;
    if (int rc = launch_gemm(ctx, EPI_BIAS_ACT, fc_tile(rows), h1, NET_H1, w2b, NET_H1, g, 1, st)) return rc;
    prof_mark(ctx, st, "fc2 forward GEMM");
    return 0;
}

}  // namespace

// ======================================================================================================
extern "C" int64_t maze_dqn_net_workspace_bytes(int max_batch) {
    if (max_batch < 1) return -1;
    return (int64_t)carve(nullptr, max_batch).bytes;
}

extern "C" int maze_dqn_gemm_bf16(maze_ctx* ctx, const uint16_t* A, int lda, const uint16_t* B, int ldb, void* C, int ldc, int M, int N, int K,
                                  int epilogue, int act, const float* bias, const uint16_t* aux, int ldaux, int tile_n, int splits, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (!A || !B || !C) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_gemm_bf16 pointer");
    if (epilogue < 0 || epilogue > 3 || act < 0 || act > 2 || (tile_n != 128 && tile_n != 256 && tile_n != 512))
        return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_gemm_bf16 epilogue / act / tile_n");
    const bool mn = epilogue == 3;   // C fp32 += A^T . B with A [K, M], B [K, N]
    if (mn) epilogue = EPI_RED_F32;
    if (epilogue == EPI_MASK && !aux) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_gemm_bf16: aux");
    GemmArgs g{};
    g.M = M; g.N = N; g.K = K; g.C = C; g.ldc = ldc; g.bias = bias; g.aux = reinterpret_cast<const bf16*>(aux); g.ldaux = ldaux; g.act = act;
    return launch_gemm(ctx, epilogue, tile_n, reinterpret_cast<const bf16*>(A), lda, reinterpret_cast<const bf16*>(B), ldb, g, splits,
                       static_cast<cudaStream_t>(stream), mn);
}

extern "C" int maze_dqn_net_refresh(maze_ctx* ctx, const maze_dqn_net* net, int which, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = check_net(ctx, net, false)) return rc;
    if (which != 0 && which != 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_net_refresh: which (0 source, 1 target)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float* p = which ? net->target : net->params;
    bf16* w1b = reinterpret_cast<bf16*>(which ? net->tw1_bf16 : net->w1_bf16);
    bf16* w2b = reinterpret_cast<bf16*>(which ? net->tw2_bf16 : net->w2_bf16);
    bf16* w1t = which ? nullptr : reinterpret_cast<bf16*>(net->w1t_bf16);
    bf16* w2t = which ? nullptr : reinterpret_cast<bf16*>(net->w2t_bf16);
    net_refresh_kernel<<<dim3(NET_IN / 32, NET_H1 / 32), 256, 0, st>>>(p + MAZE_NET_OFF_W1, NET_H1, NET_IN, w1b, w1t);
    net_refresh_kernel<<<dim3(NET_H1 / 32, NET_H2 / 32), 256, 0, st>>>(p + MAZE_NET_OFF_W2, NET_H2, NET_H1, w2b, w2t);
    net_conv_image_kernel<<<1, 256, 0, st>>>(p + MAZE_NET_OFF_CONV_W, carve(net->workspace, net->max_batch).conv_image[which]);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_dqn_features(maze_ctx* ctx, const maze_dqn_net* net, int which, const float* vec, const uint32_t* win, int n,
                                 uint16_t* X, uint8_t* pool_idx, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = check_net(ctx, net, false)) return rc;
    if (!vec || !win || !X) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_features pointer");
    if (n < 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_features: n");
    NetDropout d;
    return features(ctx, pool_idx != nullptr, vec, win, n, which ? net->target : net->params,
                    carve(net->workspace, net->max_batch).conv_image[which], reinterpret_cast<bf16*>(X), pool_idx,
                    static_cast<cudaStream_t>(stream), dropout_of(net, 3, d));
}

extern "C" int maze_dqn_forward(maze_ctx* ctx, const maze_dqn_net* net, int which, const float* vec, const uint32_t* win, int n, float* q_out,
                                void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = check_net(ctx, net, false)) return rc;
    if (!vec || !win || !q_out) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_forward pointer");
    if (n < 1 || n > net->max_batch) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_forward: n (1 .. max_batch)");
    if (which != 0 && which != 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_forward: which (0 source, 1 target)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace w = carve(net->workspace, net->max_batch);
    const float* p = which ? net->target : net->params;
    NetDropout d;
    if (int rc = features(ctx, false, vec, win, n, p, w.conv_image[which], w.X, nullptr, st, dropout_of(net, 3, d))) return rc;
    if (int rc = mlp_forward(ctx, w.X, n, reinterpret_cast<const bf16*>(which ? net->tw1_bf16 : net->w1_bf16),
                             reinterpret_cast<const bf16*>(which ? net->tw2_bf16 : net->w2_bf16), p, w.h1, w.h2, st))
        return rc;
    const int grid = (n + 7) / 8 < ctx->num_sms * 4 ? (n + 7) / 8 : ctx->num_sms * 4;
    net_head_q_kernel<<<grid, HEAD_THREADS, 0, st>>>(w.h2, n, p + MAZE_NET_OFF_W3, p + MAZE_NET_OFF_B3, q_out);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_dqn_backward(maze_ctx* ctx, const maze_dqn_net* net, const float* vec, const uint32_t* win, const float* next_vec,
                                 const uint32_t* next_win, const uint8_t* action, const float* reward, int n, float gamma, float* qsa_out,
                                 void* fc_ready_event, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = check_net(ctx, net, true)) return rc;
    if (!vec || !win || !next_vec || !next_win || !action || !reward) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_backward pointer");
    if (n < 8 || (n % 8) != 0 || n > net->max_batch) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_backward: n (multiple of 8, <= max_batch)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace w = carve(net->workspace, net->max_batch);
    const size_t np = (size_t)w.np;   // the next-state half starts at row np of X / h1 / h2
    const float* p = net->params;
    float* gr = net->grads;
    const bf16 *w1b = reinterpret_cast<const bf16*>(net->w1_bf16), *w2b = reinterpret_cast<const bf16*>(net->w2_bf16);
    const bf16 *w1t = reinterpret_cast<const bf16*>(net->w1t_bf16), *w2t = reinterpret_cast<const bf16*>(net->w2t_bf16);
    prof_reset(ctx, st);
    MAZE_CHECK(cudaMemsetAsync(net->loss, 0, sizeof(float), st));
    // forward: source net on states and next states (double-Q only: the DQN target does not need it), target net on next
    // states; with dropout each forward draws its own mask, and the saved pool choices are forward 0's
    bf16* Xt = w.dX;   // the target net has its own conv weights, so its own features; dX is free until the backward-data GEMM
    const bf16 *tw1b = reinterpret_cast<const bf16*>(net->tw1_bf16), *tw2b = reinterpret_cast<const bf16*>(net->tw2_bf16);
    const bool double_q = net->update == 0;
    NetDropout d[3];
    const NetDropout* drop0 = dropout_of(net, 0, d[0]);
    if (int rc = features(ctx, true, vec, win, n, p, w.conv_image[0], w.X, w.idx, st, drop0)) return rc;
    if (int rc = mlp_forward(ctx, w.X, n, w1b, w2b, p, w.h1, w.h2, st)) return rc;
    if (double_q) {
        if (int rc = features(ctx, false, next_vec, next_win, n, p, w.conv_image[0], w.X + np * NET_IN, nullptr, st, dropout_of(net, 1, d[1]))) return rc;
        if (int rc = mlp_forward(ctx, w.X + np * NET_IN, n, w1b, w2b, p, w.h1 + np * NET_H1, w.h2 + np * NET_H2, st)) return rc;
    }
    if (int rc = features(ctx, false, next_vec, next_win, n, net->target, w.conv_image[1], Xt, nullptr, st, dropout_of(net, 2, d[2]))) return rc;
    if (int rc = mlp_forward(ctx, Xt, n, tw1b, tw2b, net->target, w.h1t_tn, w.h2_tn, st)) return rc;
    {
        const int grid = (n + 7) / 8 < 2 * ctx->num_sms ? (n + 7) / 8 : 2 * ctx->num_sms;   // two CTAs per SM; the fc3 gradient is merged with one atomic per CTA and entry
        const auto head = double_q ? net_head_loss_kernel<UPDATE_DOUBLE_Q> : net_head_loss_kernel<UPDATE_MAX_TARGET>;
        MAZE_CHECK(cudaFuncSetAttribute(head, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HEAD_LOSS_SMEM));
        head<<<grid, HEAD_THREADS, HEAD_LOSS_SMEM, st>>>(w.h2, double_q ? w.h2 + np * NET_H2 : nullptr, w.h2_tn, n, p + MAZE_NET_OFF_W3, p + MAZE_NET_OFF_B3,
                                                         net->target + MAZE_NET_OFF_W3, net->target + MAZE_NET_OFF_B3, action, reward, gamma,
                                                         w.dh2, gr + MAZE_NET_OFF_W3, gr + MAZE_NET_OFF_B3, net->loss, qsa_out);
        MAZE_CHECK(cudaGetLastError());
        prof_mark(ctx, st, double_q ? "head: Q, double-Q target, loss, dQ, fc3 gradients" : "head: Q, max target, loss, dQ, fc3 gradients");
    }
    // fc2: dW2 = dh2^T . h1 (MN-major operands: straight from the [n, features] activations), db2 = colsum(dh2),
    //      dh1 = (dh2 . W2) * LeakyReLU'(h1)
    const int nkb_n = (n + BK - 1) / BK;
    net_colsum_kernel<<<dim3(NET_H2 / COLSUM_COLS, (n + COLSUM_ROWS - 1) / COLSUM_ROWS), 256, 0, st>>>(w.dh2, n, NET_H2, NET_H2, gr + MAZE_NET_OFF_B2);
    MAZE_CHECK(cudaGetLastError());
    prof_mark(ctx, st, "fc2 bias gradient (column sums)");
    GemmArgs g{};
    g.M = NET_H2; g.N = NET_H1; g.K = n; g.C = gr + MAZE_NET_OFF_W2; g.ldc = NET_H1;
    if (int rc = launch_gemm(ctx, EPI_RED_F32, 256, w.dh2, NET_H2, w.h1, NET_H1, g, auto_splits((NET_H2 / BM) * (NET_H1 / 256), nkb_n, ctx->num_sms), st, true)) return rc;
    prof_mark(ctx, st, "fc2 weight gradient GEMM (split-K)");
    g = GemmArgs{};
    g.M = n; g.N = NET_H1; g.K = NET_H2; g.C = w.dh1; g.ldc = NET_H1; g.aux = w.h1; g.ldaux = NET_H1; g.act = ACT_LRELU;
    if (int rc = launch_gemm(ctx, EPI_MASK, fc_tile(n), w.dh2, NET_H2, w2t, NET_H2, g, 1, st)) return rc;
    prof_mark(ctx, st, "fc2 backward-data GEMM (masked)");
    // fc1: dW1 = dh1^T . X, db1 = colsum(dh1), dX = dh1 . W1
    net_colsum_kernel<<<dim3(NET_H1 / COLSUM_COLS, (n + COLSUM_ROWS - 1) / COLSUM_ROWS), 256, 0, st>>>(w.dh1, n, NET_H1, NET_H1, gr + MAZE_NET_OFF_B1);
    MAZE_CHECK(cudaGetLastError());
    prof_mark(ctx, st, "fc1 bias gradient (column sums)");
    g = GemmArgs{};
    g.M = NET_H1; g.N = NET_IN; g.K = n; g.C = gr + MAZE_NET_OFF_W1; g.ldc = NET_IN;
    if (int rc = launch_gemm(ctx, EPI_RED_F32, 256, w.dh1, NET_H1, w.X, NET_IN, g, auto_splits((NET_H1 / BM) * ((NET_IN + 255) / 256), nkb_n, ctx->num_sms), st, true)) return rc;
    prof_mark(ctx, st, "fc1 weight gradient GEMM (split-K)");
    // every gradient but the conv layer's (the first MAZE_NET_OFF_W1 floats of the flat buffer) is complete here: a caller
    // that all-reduces gradients can start on grads[MAZE_NET_OFF_W1:] while the backward-data GEMM and the conv gradient run
    if (fc_ready_event) MAZE_CHECK(cudaEventRecord(static_cast<cudaEvent_t>(fc_ready_event), st));
    g = GemmArgs{};
    g.M = n; g.N = NET_CONV_OUT; g.K = NET_H1; g.C = w.dX; g.ldc = NET_IN; g.act = ACT_NONE;
    if (int rc = launch_gemm(ctx, EPI_BIAS_ACT, fc_tile(n), w.dh1, NET_H1, w1t, NET_H1, g, 1, st)) return rc;
    prof_mark(ctx, st, "fc1 backward-data GEMM");
    {
        const auto conv_bwd = drop0 ? net_conv_bwd_tc_kernel<true> : net_conv_bwd_tc_kernel<false>;
        MAZE_CHECK(cudaFuncSetAttribute(conv_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CB_SMEM));
        const int grid = n < ctx->num_sms * 3 ? n : ctx->num_sms * 3;   // 48 KB of operands + 9 KB of staging per CTA: three fit an SM
        conv_bwd<<<grid, CB_THREADS, CB_SMEM, st>>>(w.dX, w.idx, win, n, gr + MAZE_NET_OFF_CONV_W, gr + MAZE_NET_OFF_CONV_B, drop0 ? drop0->scale : 1.f);
        MAZE_CHECK(cudaGetLastError());
    }
    prof_mark(ctx, st, "conv gradient (un-pool + implicit GEMM)");
    return 0;
}

void maze_net_profile_free(maze_ctx* ctx) {   // called by maze_ctx_destroy
    NetProfile* pr = static_cast<NetProfile*>(ctx->net_profile);
    if (!pr) return;
    for (auto& e : pr->ev)
        if (e) cudaEventDestroy(e);
    delete pr;
    ctx->net_profile = nullptr;
}

extern "C" int maze_dqn_net_profile(maze_ctx* ctx, int enable) {
    if (!ctx) return MAZE_E_NULL;
    if (!ctx->net_profile) ctx->net_profile = new NetProfile();
    NetProfile* pr = static_cast<NetProfile*>(ctx->net_profile);
    pr->on = enable != 0;
    pr->count = 0;
    return 0;
}

extern "C" int maze_dqn_net_profile_read(maze_ctx* ctx, float* ms, char* labels, int label_bytes, int cap, int* count) {
    if (!ctx) return MAZE_E_NULL;
    if (!ms || !count || cap < 0 || (labels && label_bytes < 1)) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_net_profile_read arguments");
    NetProfile* pr = static_cast<NetProfile*>(ctx->net_profile);
    *count = 0;
    if (!pr || pr->count < 2) return 0;
    MAZE_CHECK(cudaEventSynchronize(pr->ev[pr->count - 1]));
    for (int i = 1; i < pr->count && i - 1 < cap; ++i) {
        MAZE_CHECK(cudaEventElapsedTime(&ms[i - 1], pr->ev[i - 1], pr->ev[i]));
        if (labels) {
            strncpy(labels + (size_t)(i - 1) * label_bytes, pr->label[i], (size_t)label_bytes - 1);
            labels[(size_t)(i - 1) * label_bytes + label_bytes - 1] = 0;
        }
        *count = i;
    }
    return 0;
}

extern "C" int maze_dqn_adamw(maze_ctx* ctx, const maze_dqn_net* net, float lr, float beta1, float beta2, float eps, float weight_decay,
                              int64_t step, float grad_scale, float clamp, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = check_net(ctx, net, true)) return rc;
    if (step < 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_adamw: step counts from 1");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
    net_adamw_kernel<<<(MAZE_NET_PARAMS / 4 + 255) / 256, 256, 0, st>>>(net->params, net->grads, net->adam_m, net->adam_v, (int)MAZE_NET_PARAMS, lr, beta1,
                                                                       beta2, eps, weight_decay, bc1, sqrtf(bc2), grad_scale, clamp);
    MAZE_CHECK(cudaGetLastError());
    return maze_dqn_net_refresh(ctx, net, 0, stream);
}

extern "C" int maze_dqn_sample_packed(maze_ctx* ctx, const maze_replay* r, int n, uint64_t seed, uint64_t draw, float* vec, uint32_t* win,
                                      float* next_vec, uint32_t* next_win, uint8_t* action, float* reward, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (!r || !r->pushed || !r->vec || !r->next_vec || !r->win || !r->next_win || !r->action || !r->reward)
        return maze_fail_arg(ctx, MAZE_E_NULL, "replay pointer");
    if (n < 1 || r->capacity < 1) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_dqn_sample_packed: n / capacity");
    if (!vec || !win || !next_vec || !next_win || !action || !reward) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_dqn_sample_packed output");
    net_sample_packed_kernel<<<(n + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(*r, n, seed, draw, vec, win, next_vec, next_win, action, reward);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}
