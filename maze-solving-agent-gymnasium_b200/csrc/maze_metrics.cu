// maze_difficulty: McClendon difficulty / complexity and Kim-Crawfis L / DE / D of mazes whose
// block grids live in a pool, one CTA per maze.  Toroidal (border-less) slots are scored on the
// zero-padded grid, which is exactly the bordered maze gen_maze_no_border scored before stripping
// (lib/maze_generation.py:48-56; trainers pad the same way, off_policy_trainer.py:63-64).
#include "maze_metrics.cuh"
#include "maze_walls.cuh"

namespace {

__global__ void __launch_bounds__(METRIC_THREADS)
maze_difficulty_kernel(const uint8_t* __restrict__ grids, const int32_t* __restrict__ meta,
                       const int32_t* __restrict__ ids, int n, int slot, int smem_hw, int smem_cells,
                       double* __restrict__ out, double* __restrict__ ext_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ MazeMetrics s_out;
    const int tid = threadIdx.x;
    FieldSmem f = field_smem_carve(smem, smem_hw);
    MetricsSmem ms = metrics_smem_carve(smem + field_smem_bytes(smem_hw), smem_cells, f.queue);
    for (int item = blockIdx.x; item < n; item += gridDim.x) {
        const int m = ids ? ids[item] : item;
        const int32_t* mm = meta + (size_t)m * MAZE_META_WORDS;
        const int H = mm[MAZE_META_H], W = mm[MAZE_META_W];
        const int start = mm[MAZE_META_START], goal = mm[MAZE_META_GOAL];
        const int pad = (mm[MAZE_META_FLAGS] & MAZE_FLAG_TOROIDAL) ? 1 : 0;
        const int Hb = H + 2 * pad, Wb = W + 2 * pad;
        const uint8_t* g = grids + (size_t)m * slot;
        __syncthreads();
        for (int i = tid; i < Hb * Wb; i += METRIC_THREADS) {
            const int r = i / Wb - pad, c = i % Wb - pad;
            f.grid[i] = (r >= 0 && r < H && c >= 0 && c < W) ? g[r * W + c] : 0;
        }
        __syncthreads();
        const int start_idx = ((start & 0xffff) + pad) * Wb + (start >> 16) + pad;
        const int goal_idx = ((goal & 0xffff) + pad) * Wb + (goal >> 16) + pad;
        // block distances from start: bit-parallel BFS over the cell lattice by warp 0 (one level per
        // cell distance, whatever the frontier size); lattices above 64 x 64 cells use the CTA-wide BFS
        const int nr = (Hb - 1) / 2, nc = (Wb - 1) / 2;
        if (nr <= MAZE_GEN_MAX_CELLS && nc <= MAZE_GEN_MAX_CELLS && (start_idx / Wb & 1) && (start_idx % Wb & 1)) {
            for (int i = tid; i < Hb * Wb; i += METRIC_THREADS) f.dist[i] = DIST_INF;
            __syncthreads();
            if (tid < 32) {
                Walls w;
                walls_from_grid(f.grid, Wb, nr, nc, w);
                cell_bfs_distances(w, (start_idx / Wb - 1) >> 1, (start_idx % Wb - 1) >> 1, f.dist, Wb);
            }
            __syncthreads();
        } else {
            block_bfs(f, Hb, Wb, false, start_idx);
        }
        maze_metrics(f, ms, Hb, Wb, start_idx, goal_idx, s_out, true, ext_out != nullptr);
        if (ext_out && tid < MAZE_METRIC_EXT_WORDS) ext_out[(size_t)item * MAZE_METRIC_EXT_WORDS + tid] = s_out.ext[tid];
        if (tid == 0) {
            double* o = out + (size_t)item * MAZE_METRIC_WORDS;
            o[MAZE_METRIC_DIFFICULTY] = s_out.difficulty;
            o[MAZE_METRIC_COMPLEXITY] = s_out.complexity;
            o[MAZE_METRIC_L] = s_out.L;
            o[MAZE_METRIC_DE] = s_out.DE;
            o[MAZE_METRIC_D] = s_out.D;
            o[MAZE_METRIC_SOL_LEN] = (double)s_out.sol_len;
            o[MAZE_METRIC_DE_COUNT] = (double)s_out.de_count;
            o[7] = 0.0;
        }
    }
}

}  // namespace

static int launch_difficulty(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids,
                             int n, int slot, int max_h, int max_w, double* out, double* ext_out, void* stream) {
    if (!grids || !meta || !out) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_difficulty pointer");
    if (n <= 0 || slot <= 0) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_difficulty n / slot");
    if (max_h < 5 || max_w < 5 || !(max_h & 1) || !(max_w & 1) || max_h + 2 > MAZE_GEN_MAX_DIM || max_w + 2 > MAZE_GEN_MAX_DIM)
        return maze_fail_arg(ctx, MAZE_E_SHAPE, "maze_difficulty: max shape must be odd, >= 5 and <= MAZE_GEN_MAX_DIM - 2");
    if (max_h * max_w > slot) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_difficulty: slot smaller than max shape");
    const int smem_hw = (max_h + 2) * (max_w + 2);
    const int smem_cells = ((max_h + 1) / 2) * ((max_w + 1) / 2);
    const size_t smem = field_smem_bytes(smem_hw) + metrics_smem_bytes(smem_cells);
    MAZE_CHECK(cudaFuncSetAttribute(maze_difficulty_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    MAZE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, maze_difficulty_kernel, METRIC_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    const int resident = per_sm * (ctx->num_sms > 0 ? ctx->num_sms : 148);
    maze_difficulty_kernel<<<n < resident ? n : resident, METRIC_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(
        grids, meta, ids, n, slot, smem_hw, smem_cells, out, ext_out);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_difficulty(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids,
                               int n, int slot, int max_h, int max_w, double* out, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    return launch_difficulty(ctx, grids, meta, ids, n, slot, max_h, max_w, out, nullptr, stream);
}

extern "C" int maze_difficulty_ext(maze_ctx* ctx, const uint8_t* grids, const int32_t* meta, const int32_t* ids,
                                   int n, int slot, int max_h, int max_w, double* out, double* ext_out, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (!ext_out) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_difficulty_ext: ext_out");
    return launch_difficulty(ctx, grids, meta, ids, n, slot, max_h, max_w, out, ext_out, stream);
}
