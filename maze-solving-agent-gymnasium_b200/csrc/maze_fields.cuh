// Per-maze fields shared by maze_fields (grids uploaded by the caller) and the generators:
// block-level BFS from the goal in shared memory, then the one-byte-per-block step table and the
// step budget.  One CTA per maze.
#pragma once
#include "maze_common.cuh"

constexpr int FIELD_THREADS = 128;    // maze_fields / toroidal fields kernels (block BFS: barrier-bound)
// maze_difficulty and the scored generation kernel (latency-bound pointer walks).  128 .. 512 measured on B200:
// 384 = 3 CTAs x 12 warps per SM is the best for maze_difficulty.
constexpr int METRIC_THREADS = 384;
constexpr unsigned short DIST_INF = 0xffffu;

struct FieldSmem {
    uint8_t* grid;          // [HW] 0 wall / !=0 open
    unsigned short* dist;   // [HW]
    unsigned short* queue;  // [HW]
};

__host__ __device__ inline size_t field_smem_bytes(int hw) {
    size_t g = ((size_t)hw + 15) & ~(size_t)15;
    size_t d = (((size_t)hw * 2) + 15) & ~(size_t)15;
    return g + 2 * d;
}

__device__ inline FieldSmem field_smem_carve(unsigned char* base, int hw) {
    FieldSmem f;
    size_t g = ((size_t)hw + 15) & ~(size_t)15;
    size_t d = (((size_t)hw * 2) + 15) & ~(size_t)15;
    f.grid = base;
    f.dist = reinterpret_cast<unsigned short*>(base + g);
    f.queue = reinterpret_cast<unsigned short*>(base + g + d);
    return f;
}

// Level-synchronous BFS over the block graph from `src` (block index).  Narrow frontiers
// (<= 32 blocks: every level of a dfs maze) are advanced by warp 0 alone with warp-level
// synchronisation; wide ones by the whole CTA.  All threads of the CTA must call this.
// Result: f.dist[i] = distance in blocks (DIST_INF if unreachable).
__device__ inline void block_bfs(const FieldSmem& f, int H, int W, bool tor, int src) {
    __shared__ int s_lo, s_hi, s_tail, s_level;
    const int tid = threadIdx.x;
    const int hw = H * W;
    for (int i = tid; i < hw; i += blockDim.x) f.dist[i] = DIST_INF;
    __syncthreads();
    if (tid == 0) {
        f.dist[src] = 0;
        f.queue[0] = (unsigned short)src;
        s_lo = 0; s_hi = 1; s_tail = 1; s_level = 0;
    }
    auto expand = [&](int node, int level) {
        const int r = node / W, c = node - r * W;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int nr = r + (k == 1) - (k == 0), nc = c + (k == 3) - (k == 2);
            if (tor) {
                nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
                nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
            } else if (nr < 0 || nr >= H || nc < 0 || nc >= W) {
                continue;
            }
            const int ni = nr * W + nc;
            if (f.grid[ni] != 0 && f.dist[ni] == DIST_INF) {
                // several frontier blocks may reach ni in the same level: claim it once
                unsigned short* word = f.dist + ni;
                unsigned int* aligned = reinterpret_cast<unsigned int*>(reinterpret_cast<uintptr_t>(word) & ~(uintptr_t)3);
                const bool hi = (reinterpret_cast<uintptr_t>(word) & 2) != 0;
                unsigned int old = *aligned, assumed;
                bool won = false;
                do {
                    assumed = old;
                    unsigned short cur = hi ? (unsigned short)(assumed >> 16) : (unsigned short)(assumed & 0xffff);
                    if (cur != DIST_INF) break;
                    unsigned int repl = hi ? ((assumed & 0x0000ffffu) | ((unsigned int)(level + 1) << 16))
                                           : ((assumed & 0xffff0000u) | (unsigned int)(level + 1));
                    old = atomicCAS(aligned, assumed, repl);
                    won = (old == assumed);
                } while (!won);
                if (won) f.queue[atomicAdd(&s_tail, 1)] = (unsigned short)ni;
            }
        }
    };
    for (;;) {
        __syncthreads();
        const int lo = s_lo, hi = s_hi;
        if (lo >= hi) break;
        if (hi - lo <= 32) {
            if (tid < 32) {
                int wlo = lo, whi = hi, level = s_level;
                while (wlo < whi && whi - wlo <= 32) {
                    if (wlo + tid < whi) expand(f.queue[wlo + tid], level);
                    __syncwarp();
                    wlo = whi;
                    whi = *((volatile int*)&s_tail);
                    ++level;
                    __syncwarp();
                }
                if (tid == 0) { s_lo = wlo; s_hi = whi; s_level = level; }
            }
        } else {
            const int level = s_level;
            for (int i = lo + tid; i < hi; i += blockDim.x) expand(f.queue[i], level);
            __syncthreads();
            if (tid == 0) { s_lo = hi; s_hi = s_tail; s_level = level + 1; }
        }
    }
    __syncthreads();
}

// simple_maze_env.py:52-58 + metrics_calculator.py:16,22-26, evaluated in IEEE double with the
// same operation order (divide, multiply, ceil; no contraction).
__device__ inline int max_steps_budget(int H, int W, int sol_len) {
    const double ce = (double)((H - 1) * ((W - 1) / 2) - 1);
    const double factor = __ddiv_rn((double)sol_len, ce);
    return (int)ceil(__dmul_rn((double)((H - 1) * (W - 1) - 1), factor));
}

// Step table from the goal-distance field (closed form of base_maze_env.py:224-262, see
// oracle/grid.py:best_dir_code_table).  All threads of the CTA call this after block_bfs.
__device__ inline void encode_step_table(const FieldSmem& f, int H, int W, bool tor, int goal_r, int goal_c,
                                         uint8_t* __restrict__ out) {
    const int hw = H * W;
    const int L = 2 * (H < W ? H : W);
    for (int i = threadIdx.x; i < hw; i += blockDim.x) {
        if (f.grid[i] == 0) { out[i] = 0; continue; }   // walls carry no step information
        const int r = i / W, c = i - r * W;
        int best = 0x7fffffff, code = 4;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            int dr, dc;
            action_delta(a, dr, dc);
            int nr = r + dr, nc = c + dc;
            if (tor) {
                nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
                nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
            } else if (!(nr > 0 && nr < H && nc > 0 && nc < W)) {   // simple_maze_env.py:68
                continue;
            }
            const int ni = nr * W + nc;
            if (f.grid[ni] == 0) continue;
            const int d = f.dist[ni];
            if (d == DIST_INF) continue;
            const int p = (d < L ? d : L) + 1;
            const int score = 20 * p + 3 * (abs(nr - goal_r) + abs(nc - goal_c));
            if (score < best) { best = score; code = a; }
        }
        const int d = f.dist[i];
        const int d4 = (d == DIST_INF) ? 0 : (d & 3);
        out[i] = (uint8_t)((f.grid[i] != 0 ? MAZE_TAB_OPEN : 0) | (code << MAZE_TAB_CODE_SHIFT) | (d4 << MAZE_TAB_D4_SHIFT));
    }
}

// Fields of the maze in slot m whose block grid lies in global memory: BFS from the goal, step table,
// step budget (the body of maze_fields; also the second half of toroidal generation).  One CTA.
__device__ inline void fields_of_slot(const FieldSmem& f, const uint8_t* __restrict__ grids, int32_t* __restrict__ meta,
                                      uint8_t* __restrict__ table, int m, int slot) {
    int32_t* mm = meta + (size_t)m * MAZE_META_WORDS;
    const int H = mm[MAZE_META_H], W = mm[MAZE_META_W];
    const int start = mm[MAZE_META_START], goal = mm[MAZE_META_GOAL];
    const bool tor = (mm[MAZE_META_FLAGS] & MAZE_FLAG_TOROIDAL) != 0;
    const uint8_t* g = grids + (size_t)m * slot;
    __syncthreads();
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) f.grid[i] = g[i];
    __syncthreads();
    const int gr = goal & 0xffff, gc = goal >> 16;
    block_bfs(f, H, W, tor, gr * W + gc);
    encode_step_table(f, H, W, tor, gr, gc, table + (size_t)m * slot);
    if (threadIdx.x == 0) {
        const int d = f.dist[(start & 0xffff) * W + (start >> 16)];
        const int sol_len = (d == DIST_INF) ? 0 : d + 1;
        mm[MAZE_META_SOL_LEN] = sol_len;
        mm[MAZE_META_MAX_STEPS] = max_steps_budget(H, W, sol_len);
    }
}
