// Enriched (-v1) observation and direction-mask kernels (sm_100a).
//
// maze_window: one warp per env writes the float32 [3, 15, 15] crop around the agent
// (lib/maze_handler.py:4-99) -- 2 700 B of coalesced streaming stores per env; the maze comes from
// the L2-resident step table, the visited state from the env's visit bitmap or visit counters.
// HBM-write bound.
// maze_direction_mask: one thread per env, four table bytes (lib/maze_handler.py:122-162,
// simple_maze_env.py:41-50, toroidal_maze_env.py:57-70).
#include "maze_env.cuh"
#include "maze_window.cuh"

namespace {

constexpr int OBS_THREADS = 256;
constexpr int WIN = MAZE_WINDOW;
constexpr int WIN_CELLS = WIN * WIN;

// A CTA of 256 threads serves 16 consecutive envs, 16 lanes each: lane r < 15 owns window row r and assembles its three
// 15-bit masks in registers (window_row_masks: 15 table bytes + 15 visit words per lane; a 4 x 4 visit tile is one
// 32-byte sector shared by the four lanes whose rows cross it), then writes them as bytes into shared memory, laid out
// exactly like the output; then all 256 threads stream the 16 x 2 700 bytes out as 16-byte stores, four shared bytes ->
// one float4 (16 envs x 675 floats start on a 16-byte boundary; one env's 2 700 bytes do not).  History (ncu): first
// version 1 080 warp instructions per env (one 4-byte store per value, div / mod per block); round 1's warp-per-env
// gather 757, issue slots 78 % busy at 0.48 of the HBM peak (profiles/r01j_window_after_details.txt); this one-lane-
// per-row form does the gather in about a quarter of the instructions.
constexpr int WIN_ENVS = OBS_THREADS / 16;
constexpr int WIN_FLOATS = 3 * WIN_CELLS;

constexpr int WIN_MIN_BLOCKS = 4;   // __launch_bounds__ of both window kernels

// masks of one window row -> the row's 3 x 15 output bytes in shared memory
__device__ __forceinline__ void window_row_to_smem(uint8_t* sl, unsigned m0, unsigned m1, unsigned m2) {
#pragma unroll
    for (int j = 0; j < WIN; ++j) {
        sl[j] = (uint8_t)((m0 >> j) & 1u);
        sl[WIN_CELLS + j] = (uint8_t)((m1 >> j) & 1u);
        sl[2 * WIN_CELLS + j] = (uint8_t)((m2 >> j) & 1u);
    }
}

__device__ __forceinline__ void window_norms(const EnvState& st, const MazeView& mz, int e, int hl, double* __restrict__ agent_norm,
                                             double* __restrict__ target_norm) {
    if (hl < 2) {
        const double shape = (double)(hl == 0 ? mz.H : mz.W);
        if (agent_norm) agent_norm[(size_t)e * 2 + hl] = __ddiv_rn((double)(hl == 0 ? st.r : st.c), shape);
        if (target_norm) target_norm[(size_t)e * 2 + hl] = __ddiv_rn((double)(hl == 0 ? (mz.goal & 0xffff) : (mz.goal >> 16)), shape);
    }
}

// all threads of the CTA: `n_envs` x 2 700 bytes of shared memory -> float32 in global memory, 16 bytes per store
__device__ __forceinline__ void window_stream_out(const uint8_t* s_out, float* __restrict__ out, int n_float) {
    for (int q = threadIdx.x; 4 * q < n_float; q += OBS_THREADS) {
        const int f = 4 * q;
        const unsigned v = *reinterpret_cast<const unsigned*>(s_out + f);   // four values, one byte each
        if (f + 3 < n_float) {
            __stcs(reinterpret_cast<float4*>(out) + q,
                   make_float4(__uint_as_float((v & 1u) * 0x3f800000u), __uint_as_float((v >> 8 & 1u) * 0x3f800000u),
                               __uint_as_float((v >> 16 & 1u) * 0x3f800000u), __uint_as_float((v >> 24 & 1u) * 0x3f800000u)));
        } else {
            for (int i = f; i < n_float; ++i) __stcs(out + i, (float)s_out[i]);
        }
    }
}

__global__ void __launch_bounds__(OBS_THREADS, WIN_MIN_BLOCKS)
maze_window_kernel(maze_env_batch b, float* __restrict__ window, double* __restrict__ agent_norm,
                   double* __restrict__ target_norm) {
    __shared__ __align__(16) uint8_t s_out[WIN_ENVS * WIN_FLOATS];
    const int hl = threadIdx.x & 15, w = threadIdx.x >> 4;
    const int e0 = blockIdx.x * WIN_ENVS, e = e0 + w;
    if (e < b.num_envs) {
        const EnvState st = unpack_state(b.state[e]);
        const MazeView mz = load_maze(b, b.env_maze[e]);
        unsigned m0, m1, m2;
        window_row_masks(b, e, st, mz, hl, m0, m1, m2);
        if (hl < WIN) window_row_to_smem(s_out + w * WIN_FLOATS + hl * WIN, m0, m1, m2);   // block (row, col) of channel ch is output index 225 ch + 15 row + col
        window_norms(st, mz, e, hl, agent_norm, target_norm);
    }
    __syncthreads();
    window_stream_out(s_out, window + (size_t)e0 * WIN_FLOATS, min(WIN_ENVS, b.num_envs - e0) * WIN_FLOATS);   // 16-byte aligned: e0 is a multiple of 16
}

// Bordered mazes with the visit bitmap (maze_env_batch.flags & MAZE_BATCH_BORDERED): the gather is a chain of dependent
// loads (state -> maze record -> rows), and at four CTAs per SM its latency, not HBM, paced the kernel (each CTA spends
// about 3 us in the chain before it can write its 43 KB).  Here every half-warp carries TWO envs through the chain, each
// level issued for both before either is consumed: 32 envs per CTA, twice the loads in flight at the same occupancy.
constexpr int WINB_PER = 2;   // 4 measured slower (4.7 vs 5.2 TB/s at 262 144 envs: fewer CTAs per SM by shared memory)
constexpr int WINB_ENVS = WIN_ENVS * WINB_PER;

__global__ void __launch_bounds__(OBS_THREADS, WIN_MIN_BLOCKS)
maze_window_bordered_kernel(maze_env_batch b, float* __restrict__ window, double* __restrict__ agent_norm,
                            double* __restrict__ target_norm) {
    __shared__ __align__(16) uint8_t s_out[WINB_ENVS * WIN_FLOATS];
    const int hl = threadIdx.x & 15, w = threadIdx.x >> 4;
    const int e0 = blockIdx.x * WINB_ENVS;
    int e[WINB_PER];
    bool valid[WINB_PER];
    uint64_t raw[WINB_PER];
    int maze_id[WINB_PER];
#pragma unroll
    for (int u = 0; u < WINB_PER; ++u) {
        e[u] = e0 + w * WINB_PER + u;
        valid[u] = e[u] < b.num_envs;
        raw[u] = valid[u] ? b.state[e[u]] : 0ull;
        maze_id[u] = valid[u] ? b.env_maze[e[u]] : 0;
    }
    EnvState st[WINB_PER];
    MazeView mz[WINB_PER];
#pragma unroll
    for (int u = 0; u < WINB_PER; ++u) {
        st[u] = unpack_state(raw[u]);
        mz[u] = MazeView{};
        if (valid[u]) mz[u] = load_maze(b, maze_id[u]);
    }
    WindowRowRaw rows[WINB_PER];
    bool has[WINB_PER];
#pragma unroll
    for (int u = 0; u < WINB_PER; ++u) {
        has[u] = valid[u] && hl < WIN && mz[u].H >= WIN && mz[u].W >= WIN;   // smaller mazes have no window: zeros, as in window_row_masks
        rows[u] = WindowRowRaw{};
        if (has[u]) rows[u] = window_row_load_bits(b, e[u], st[u], mz[u], hl);
    }
#pragma unroll
    for (int u = 0; u < WINB_PER; ++u) {
        if (!valid[u]) continue;
        unsigned m0 = 0, m1 = 0, m2 = 0;
        if (has[u]) window_row_fold_bits(rows[u], mz[u], m0, m1, m2);
        if (hl < WIN) window_row_to_smem(s_out + (w * WINB_PER + u) * WIN_FLOATS + hl * WIN, m0, m1, m2);
        window_norms(st[u], mz[u], e[u], hl, agent_norm, target_norm);
    }
    __syncthreads();
    window_stream_out(s_out, window + (size_t)e0 * WIN_FLOATS, min(WINB_ENVS, b.num_envs - e0) * WIN_FLOATS);
}

__global__ void __launch_bounds__(OBS_THREADS)
maze_direction_mask_kernel(maze_env_batch b, int probs, float4* __restrict__ mask) {
    const int e = blockIdx.x * OBS_THREADS + threadIdx.x;
    if (e >= b.num_envs) return;
    const EnvState st = unpack_state(b.state[e]);
    const int m = b.env_maze[e];
    const int2 shape = __ldg(reinterpret_cast<const int2*>(b.meta + (size_t)m * MAZE_META_WORDS));
    const int H = shape.x, W = shape.y;
    const bool tor = (__ldg(b.meta + (size_t)m * MAZE_META_WORDS + MAZE_META_FLAGS) & MAZE_FLAG_TOROIDAL) != 0;
    const uint8_t* tab = b.table + (size_t)m * b.slot;
    float v[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int dr, dc;
        action_delta(a, dr, dc);
        int nr = st.r + dr, nc = st.c + dc;
        bool open;
        if (tor) {
            nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
            nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
            open = (__ldg(tab + nr * W + nc) & MAZE_TAB_OPEN) != 0;
        } else {   // agents stand on interior blocks of a bordered maze; stay in the slot regardless
            open = nr >= 0 && nr < H && nc >= 0 && nc < W && (__ldg(tab + nr * W + nc) & MAZE_TAB_OPEN) != 0;
        }
        v[a] = open ? 1.0f : 0.0f;
    }
    if (probs && ((st.flags >> MAZE_ST_NMOVES_SHIFT) & 3) >= 2) {   // len(visited_cell) > 1
        const int last = (st.flags >> MAZE_ST_MOVE_SHIFT) & 3;
        // euclid: previous - current = -ACTIONS[last] -> the opposite action.  torus: the tuple is
        // built (dx, dy), i.e. column-first, before the same index lookup (toroidal_maze_env.py:63-68)
        const int back = tor ? 3 - last : (last ^ 1);
        v[back] = 0.25f;
    }
    mask[e] = make_float4(v[0], v[1], v[2], v[3]);
}

// maze_render: the frame MazeViewTemplate keeps on its pygame surface (lib/maze_view.py:12-14,88-104,
// 148-152), as uint8 [n, out_h, out_w, 3] for n selected envs.  One CTA per (env, tile row); a thread
// produces four pixels (12 bytes) at a time.
//   tile (r, c) = 16 x 16 pixels at (16 c, 16 r): CELL_COLORS[maze[r][c]] with a one-pixel outline,
//   (59, 66, 82) as drawn by __draw_maze, (208, 135, 112) once the agent has left the block
//   (_draw_cell, called by move_agent / _reset_agent on the block the agent leaves);
//   agent = 8 x 8 square at offset (4, 4) of its tile; the layers are one pixel smaller than the
//   window (:41-44), so the last pixel row / column stay black, like everything beyond the maze.
// "Left" is derived from the episode's visit counters: start once the episode has a legal move, the
// agent's own block when it is there for at least the second time, any other block with a visit.
__global__ void __launch_bounds__(OBS_THREADS)
maze_render_kernel(maze_env_batch b, const int32_t* __restrict__ env_ids, int out_h, int out_w, uint8_t* __restrict__ out) {
    constexpr int T = MAZE_RENDER_TILE;
    const int k = blockIdx.x, r = blockIdx.y;
    const int e = env_ids ? env_ids[k] : k;
    const EnvState st = unpack_state(b.state[e]);
    const int m = b.env_maze[e];
    const int4 m0 = __ldg(reinterpret_cast<const int4*>(b.meta + (size_t)m * MAZE_META_WORDS));
    const int H = m0.x, W = m0.y;
    const int start_r = m0.z & 0xffff, start_c = m0.z >> 16, goal_r = m0.w & 0xffff, goal_c = m0.w >> 16;
    const uint8_t* tab = b.table + (size_t)m * b.slot;
    const bool has_moved = ((st.flags >> MAZE_ST_NMOVES_SHIFT) & 3) >= 1;
    __shared__ uint8_t s_tile[MAZE_GEN_MAX_DIM];   // per tile of this row: value (0 / 1 / 2) | trail << 2
    for (int c = threadIdx.x; c < out_w / T; c += OBS_THREADS) {
        int code = 0;
        if (r < H && c < W) {
            const bool open = (__ldg(tab + r * W + c) & MAZE_TAB_OPEN) != 0;
            const int v = open ? ((r == goal_r && c == goal_c) ? 2 : 1) : 0;
            bool trail = false;
            if (open) {
                const unsigned vis = *VISIT_AT(b, e, visit_index(b, r, c, W));
                const int cnt = ((int)(vis >> 8) == st.epoch) ? (int)(vis & 0xff) : 0;
                if (r == start_r && c == start_c) trail = has_moved;
                else if (r == st.r && c == st.c) trail = cnt >= 2;
                else trail = cnt >= 1;
            }
            code = v | (trail ? 4 : 0) | 8;
        }
        s_tile[c] = (uint8_t)code;
    }
    __syncthreads();
    const int groups = out_w / 4;   // four pixels per thread and iteration
    for (int p = threadIdx.x; p < T * groups; p += OBS_THREADS) {
        const int ly = p / groups, x0 = (p % groups) * 4, y = r * T + ly;
        if (y >= out_h) break;
        unsigned char px[12];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int x = x0 + i, c = x / T, lx = x % T;
            const int code = s_tile[c];
            int cr = 0, cg = 0, cb = 0;
            if ((code & 8) && x != W * T - 1 && y != H * T - 1) {
                const int v = code & 3;
                if (lx == 0 || lx == T - 1 || ly == 0 || ly == T - 1) {
                    if (code & 4) { cr = 208; cg = 135; cb = 112; } else { cr = 59; cg = 66; cb = 82; }
                } else if (r == st.r && c == st.c && lx >= T / 4 && lx < T / 4 + T / 2 && ly >= T / 4 && ly < T / 4 + T / 2) {
                    cr = 94; cg = 129; cb = 172;                                     // AGENT_COLOR
                } else if (v == 0) { cr = 46; cg = 52; cb = 64; }                    // CELL_COLORS: wall, floor, goal
                else if (v == 1) { cr = 236; cg = 239; cb = 244; }
                else { cr = 163; cg = 190; cb = 140; }
            }
            px[3 * i] = (unsigned char)cr; px[3 * i + 1] = (unsigned char)cg; px[3 * i + 2] = (unsigned char)cb;
        }
        unsigned* o = reinterpret_cast<unsigned*>(out + (((size_t)k * out_h + y) * out_w + x0) * 3);
#pragma unroll
        for (int w = 0; w < 3; ++w)
            __stcs(o + w, (unsigned)px[4 * w] | ((unsigned)px[4 * w + 1] << 8) | ((unsigned)px[4 * w + 2] << 16) | ((unsigned)px[4 * w + 3] << 24));
    }
}

}  // namespace

extern "C" int maze_render(maze_ctx* ctx, const maze_env_batch* b, const int32_t* env_ids, int n, uint8_t* out,
                           int out_h, int out_w, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!out) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_render: out");
    if (n <= 0 || out_h <= 0 || out_w <= 0 || out_h % MAZE_RENDER_TILE || out_w % MAZE_RENDER_TILE ||
        out_h / MAZE_RENDER_TILE > MAZE_GEN_MAX_DIM || out_w / MAZE_RENDER_TILE > MAZE_GEN_MAX_DIM)
        return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_render: n / out_h / out_w (multiples of MAZE_RENDER_TILE, at most MAZE_GEN_MAX_DIM tiles)");
    if ((uintptr_t)out & 3) return maze_fail_arg(ctx, MAZE_E_ALIGN, "maze_render: out must be 4-byte aligned");
    if (env_ids == nullptr && n > b->num_envs) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_render: n exceeds num_envs");
    maze_render_kernel<<<dim3(n, out_h / MAZE_RENDER_TILE), OBS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*b, env_ids, out_h, out_w, out);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_window(maze_ctx* ctx, const maze_env_batch* b, float* window, double* agent_norm,
                           double* target_norm, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!window) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_window: window");
    if (((uintptr_t)window & 15) || ((uintptr_t)agent_norm & 7) || ((uintptr_t)target_norm & 7))
        return maze_fail_arg(ctx, MAZE_E_ALIGN, "maze_window pointer alignment");
    if ((b->flags & MAZE_BATCH_BORDERED) && b->visit_bits) {
        const int grid = (b->num_envs + WINB_ENVS - 1) / WINB_ENVS;
        maze_window_bordered_kernel<<<grid, OBS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*b, window, agent_norm, target_norm);
    } else {
        const int grid = (b->num_envs + WIN_ENVS - 1) / WIN_ENVS;
        maze_window_kernel<<<grid, OBS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*b, window, agent_norm, target_norm);
    }
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_direction_mask(maze_ctx* ctx, const maze_env_batch* b, int probs, float* mask, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!mask) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_direction_mask: mask");
    if ((uintptr_t)mask & 15) return maze_fail_arg(ctx, MAZE_E_ALIGN, "maze_direction_mask: mask must be 16-byte aligned");
    const int grid = (b->num_envs + OBS_THREADS - 1) / OBS_THREADS;
    maze_direction_mask_kernel<<<grid, OBS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        *b, probs, reinterpret_cast<float4*>(mask));
    MAZE_CHECK(cudaGetLastError());
    return 0;
}
