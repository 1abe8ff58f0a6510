// Env step / reset kernels (sm_100a).
//
// One env per thread (two per thread from 64 K envs up).  State is one packed 64-bit word per env
// (coalesced 8-byte load/store); the maze is read through its one-byte-per-block step table
// (L2/L1 resident for a maze pool); the only scattered DRAM access is the 2-byte visit counter of
// the block stepped onto, fetched only for legal moves, from a cell-major array.
// Every other maze_step launch runs its CTAs in reverse order, so the envs stepped last in one launch
// are stepped first in the next, while their state word, maze id and the visit counters they just
// wrote may still be in L2.  Each env's transition reads only its own data, so the order cannot
// change a result.
// Reference semantics: gymnasium_env/envs/base_maze_env.py:136-210, lib/maze_view.py:165-197.
#include "maze_env.cuh"

namespace {

constexpr int STEP_THREADS = 256;
constexpr int STEP_MIN_BLOCKS_EPT1 = 6, STEP_MIN_BLOCKS_EPT2 = 5;   // __launch_bounds__ of maze_step_kernel

// EPT environments per thread (env = base + k * STEP_THREADS keeps every access coalesced): the
// loads of all EPT envs are issued phase by phase before anything waits on them.  The dependent
// chain per env is state -> meta (L1) -> table byte (L2) -> visit counter (DRAM); the visit
// counter is only fetched when the move is legal (a wall hit needs no counter), which matters
// because every such fetch costs a whole DRAM line.
template <int EPT, bool kStats, bool kTiled>
__global__ void __launch_bounds__(STEP_THREADS, EPT == 2 ? STEP_MIN_BLOCKS_EPT2 : STEP_MIN_BLOCKS_EPT1)
maze_step_kernel(maze_env_batch b, const uint8_t* __restrict__ actions, uint32_t mode, StepLuts luts, bool reverse) {
    const int blk = reverse ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
    const int base = blk * (STEP_THREADS * EPT) + threadIdx.x;

    const uint64_t pol_state = l2_policy(), pol_table = l2_policy();
    // ---- phase 1: per-env words
    uint64_t raw[EPT];
    int m[EPT], a[EPT];
    bool valid[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        const int e = base + k * STEP_THREADS;
        valid[k] = e < b.num_envs;
        const int ee = valid[k] ? e : b.num_envs - 1;
        raw[k] = pol_load(reinterpret_cast<const unsigned long long*>(b.state) + ee, pol_state);
        m[k] = pol_load(b.env_maze + ee, pol_state);
        a[k] = __ldcs(actions + ee) & 3;
    }

    // ---- phase 2: maze metadata (L1/L2 resident: contiguous envs share a maze)
    bool do_reset[EPT];
    int hw[EPT], tor[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        const int flags = (int)((raw[k] >> 24) & 0xff);
        do_reset[k] = valid[k] && (mode & MAZE_STEP_AUTORESET) && (flags & MAZE_ST_NEEDS_RESET);
        if (do_reset[k] && (mode & MAZE_STEP_WIN_NEXT) && (flags & MAZE_ST_WON)) {
            m[k] += b.pool_stride;
            if (m[k] >= b.num_mazes) m[k] -= b.num_mazes;
            pol_store(b.env_maze + base + k * STEP_THREADS, m[k], pol_state);
        }
        const int2 shape = __ldg(reinterpret_cast<const int2*>(b.meta + (size_t)m[k] * MAZE_META_WORDS));
        hw[k] = shape.x | (shape.y << 16);
        tor[k] = __ldg(b.meta + (size_t)m[k] * MAZE_META_WORDS + MAZE_META_FLAGS) & MAZE_FLAG_TOROIDAL;
    }

    // ---- phase 3: the block stepped onto: table byte
    int npos[EPT], idx[EPT], vidx[EPT], tb[EPT];
    bool inb[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        const int H = hw[k] & 0xffff, W = hw[k] >> 16;
        const int r = (int)(raw[k] & 0xff), c = (int)((raw[k] >> 8) & 0xff);
        int dr, dc;
        action_delta(a[k], dr, dc);
        int nr = r + dr, nc = c + dc;
        if (tor[k]) {  // lib/maze_view.py:185-186
            nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
            nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
            inb[k] = true;
        } else {       // lib/maze_view.py:169
            inb[k] = (nr > 0) & (nr < H - 1) & (nc > 0) & (nc < W - 1);
        }
        if (do_reset[k]) {
            const int start = __ldg(b.meta + (size_t)m[k] * MAZE_META_WORDS + MAZE_META_START);
            nr = start & 0xffff;
            nc = start >> 16;
            inb[k] = true;
        }
        if (!inb[k]) { nr = r; nc = c; }
        npos[k] = nr | (nc << 16);
        idx[k] = nr * W + nc;
        vidx[k] = kTiled ? ((((nr >> 2) * ((W + 3) >> 2) + (nc >> 2)) << 4) | ((nr & 3) << 2) | (nc & 3)) : idx[k];
        tb[k] = pol_load_nc(b.table + (size_t)m[k] * b.slot + idx[k], pol_table);
    }

    // ---- phase 4: visit counter, only for legal moves
    const uint64_t pol = l2_policy();
    uint32_t vis[EPT];
    bool moved[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        moved[k] = valid[k] && !do_reset[k] && inb[k] && (tb[k] & MAZE_TAB_OPEN);
        vis[k] = 0;
        if (moved[k]) vis[k] = pol_load(VISIT_AT(b, base + k * STEP_THREADS, vidx[k]), pol);
    }

    // ---- phase 5: transition + outputs
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        const int e = base + k * STEP_THREADS;
        const int H = hw[k] & 0xffff, W = hw[k] >> 16;
        const int goal = __ldg(b.meta + (size_t)m[k] * MAZE_META_WORDS + MAZE_META_GOAL);
        const int max_steps = __ldg(b.meta + (size_t)m[k] * MAZE_META_WORDS + MAZE_META_MAX_STEPS);
        double reward = 0.0;
        int term = 0, trunc = 0;
        uint32_t rcode = MAZE_REC_REWARD(MAZE_REC_KIND_CONST, MAZE_REC_CONST_ZERO);   // how `reward` was obtained (packed record)
        bool wrapped = false;
        EnvState st = unpack_state(raw[k]);

        if (do_reset[k]) {
            begin_episode(st, npos[k], tb[k], wrapped);
            visit_bits_clear(b, e);
        } else if (valid[k]) {
            if (moved[k]) {
                const int cnt = ((int)(vis[k] >> 8) == st.epoch) ? (int)(vis[k] & 0xff) : 0;
                if (cnt == 0) {
                    if (npos[k] == goal) {
                        reward = 1.0;   // base_maze_env.py:185-187
                        term = 1;
                        rcode = MAZE_REC_REWARD(MAZE_REC_KIND_CONST, MAZE_REC_CONST_ONE);
                    } else {            // :189-192, len(path) = D_goal + 1
                        const int dd = ((st.tab >> MAZE_TAB_D4_SHIFT) - (tb[k] >> MAZE_TAB_D4_SHIFT)) & 3;
                        reward = dd == 1 ? luts.shaping_closer : (dd == 3 ? luts.shaping_farther : luts.shaping_same);
                        rcode = MAZE_REC_REWARD(MAZE_REC_KIND_SHAPING, dd == 1 ? 2u : (dd == 3 ? 0u : 1u));
                    }
                } else {
                    reward = __ldg(luts.revisit + cnt);   // :194
                    rcode = MAZE_REC_REWARD(MAZE_REC_KIND_REVISIT, (uint32_t)cnt);
                }
                pol_store(VISIT_AT(b, e, vidx[k]), (unsigned)((st.epoch << 8) | (cnt < 255 ? cnt + 1 : 255)), pol);   // :196
                visit_bit_set(b, e, npos[k] & 0xffff, npos[k] >> 16);
                st.r = npos[k] & 0xffff;
                st.c = npos[k] >> 16;
                st.tab = tb[k];
                st.consec = 0;
                int nm = (st.flags >> MAZE_ST_NMOVES_SHIFT) & 3;
                nm = nm < 2 ? nm + 1 : 2;
                st.flags = (a[k] << MAZE_ST_MOVE_SHIFT) | (nm << MAZE_ST_NMOVES_SHIFT);
            } else {
                st.consec = st.consec < 255 ? st.consec + 1 : 255;   // :199-200
                reward = __ldg(luts.invalid + st.consec);
                rcode = MAZE_REC_REWARD(MAZE_REC_KIND_INVALID, (uint32_t)st.consec);
                st.flags &= ~(MAZE_ST_NEEDS_RESET | MAZE_ST_WON);
            }
            st.steps = st.steps < 65535 ? st.steps + 1 : 65535;
            if (st.steps > max_steps) {   // :205-208 (overrides a goal reward on the same step)
                trunc = 1;
                reward = -1.0;
                rcode = MAZE_REC_REWARD(MAZE_REC_KIND_CONST, MAZE_REC_CONST_MINUS_ONE);
            }
            if (term | trunc) st.flags |= MAZE_ST_NEEDS_RESET | (term ? MAZE_ST_WON : 0);
        }

        // epoch wrap-around: the visit array must really be cleared (rare)
        const unsigned need = __ballot_sync(0xffffffffu, wrapped);
        if (need) warp_clear_visits(need, b, e);
        if (kStats && b.stats) {   // stats[3]: transitions made (autoreset steps are not transitions); one atomic per warp
            const unsigned stepped = __ballot_sync(0xffffffffu, valid[k] && !do_reset[k]);
            if (stepped && (threadIdx.x & 31) == 0) atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 3), (unsigned long long)__popc(stepped));
        }

        if (!valid[k]) continue;

        pol_store(reinterpret_cast<unsigned long long*>(b.state) + e, (unsigned long long)pack_state(st), pol_state);
        // `target` only changes when the env's maze does: the restart after a win (next pool maze, or the
        // regenerated slot).  The buffer persists between steps, so it is rewritten only then, and
        // target_dirty tells a host mirror that this launch touched it.
        if (do_reset[k] && (raw[k] >> 24 & MAZE_ST_WON)) {
            st_cs(reinterpret_cast<int2*>(b.target) + e, make_int2(goal & 0xffff, goal >> 16));
            if (b.target_dirty) *b.target_dirty = 1;
        }
        if (mode & MAZE_STEP_PACKED)
            __stcs(b.packed + e, (uint32_t)st.r | ((uint32_t)st.c << 8) | ((uint32_t)((st.tab >> MAZE_TAB_CODE_SHIFT) & 7) << MAZE_REC_CODE_SHIFT) |
                                     ((uint32_t)term << MAZE_REC_TERM_SHIFT) | ((uint32_t)trunc << MAZE_REC_TRUNC_SHIFT) | rcode);
        if (!(mode & MAZE_STEP_NO_WIDE)) {
            st_cs(reinterpret_cast<int2*>(b.agent) + e, make_int2(st.r, st.c));
            st_cs(reinterpret_cast<int2*>(b.best_dir) + e,
                  best_dir_from_code((st.tab >> MAZE_TAB_CODE_SHIFT) & 7, st.r, st.c, H, W, tor[k] != 0));
            st_cs(b.reward + e, reward);
            __stcs(b.terminated + e, (uint8_t)term);
            __stcs(b.truncated + e, (uint8_t)trunc);
        }

        if (kStats) {
            if (b.ep_return) {
                double g = do_reset[k] ? 0.0 : b.ep_return[e] + reward;
                b.ep_return[e] = g;
                if ((term | trunc) && b.stats_return) atomicAdd(b.stats_return, g);
            }
            if (b.stats) {
                if (term | trunc) {
                    atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 0), 1ull);
                    if (term) atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 1), 1ull);
                    else atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 2), 1ull);
                }
            }
            if (term && (mode & MAZE_STEP_WIN_QUEUE) && b.queue) {
                int at = atomicAdd(b.queue_count, 1);
                b.queue[at] = m[k];
            }
        }
    }
}

__global__ void __launch_bounds__(STEP_THREADS)
maze_reset_kernel(maze_env_batch b, const uint8_t* __restrict__ mask) {
    const int e = blockIdx.x * STEP_THREADS + threadIdx.x;
    const bool valid = e < b.num_envs;
    const int ee = valid ? e : b.num_envs - 1;
    const bool sel = valid && (mask == nullptr || mask[ee] != 0);
    bool wrapped = false;
    EnvState s;
    int H = 0, W = 0, goal = 0;
    bool tor = false;
    if (sel) {
        s = unpack_state(b.state[ee]);
        const int m = b.env_maze[ee];
        const int4* mp = reinterpret_cast<const int4*>(b.meta + (size_t)m * MAZE_META_WORDS);
        const int4 m0 = __ldg(mp);
        const int4 m1 = __ldg(mp + 1);
        H = m0.x; W = m0.y; goal = m0.w;
        tor = (m1.y & MAZE_FLAG_TOROIDAL) != 0;
        const int start = m0.z;
        const int sidx = (start & 0xffff) * W + (start >> 16);
        begin_episode(s, start, __ldg(b.table + (size_t)m * b.slot + sidx), wrapped);
        visit_bits_clear(b, ee);
    }
    const unsigned need = __ballot_sync(0xffffffffu, wrapped);
    if (need) warp_clear_visits(need, b, ee);
    if (!sel) return;
    b.state[e] = pack_state(s);
    reinterpret_cast<int2*>(b.agent)[e] = make_int2(s.r, s.c);
    reinterpret_cast<int2*>(b.target)[e] = make_int2(goal & 0xffff, goal >> 16);
    if (b.target_dirty) *b.target_dirty = 1;   // every selected thread: a masked reset need not include lane 0 (benign race)
    reinterpret_cast<int2*>(b.best_dir)[e] =
        best_dir_from_code((s.tab >> MAZE_TAB_CODE_SHIFT) & 7, s.r, s.c, H, W, tor);
    b.reward[e] = 0.0;
    b.terminated[e] = 0;
    b.truncated[e] = 0;
    if (b.ep_return) b.ep_return[e] = 0.0;
}

// k_steps transitions per env, state in registers (see maze_step_many in the header).  Same rules as
// maze_step_kernel step by step, including the next-step autoreset and the episode statistics.
__global__ void __launch_bounds__(STEP_THREADS)
maze_step_many_kernel(maze_env_batch b, const uint8_t* __restrict__ actions, int k_steps, uint32_t mode, StepLuts luts,
                      maze_step_trace tr, int e0, int e1) {
    const int e = e0 + blockIdx.x * STEP_THREADS + threadIdx.x;
    if (e >= e1) return;
    const size_t B = (size_t)b.num_envs;
    EnvState st = unpack_state(b.state[e]);
    int m = b.env_maze[e];
    MazeView mz = load_maze(b, m);
    double reward = 0.0, ep_return = b.ep_return ? b.ep_return[e] : 0.0;
    int term = 0, trunc = 0;
    bool target_changed = false;
    unsigned long long n_episodes = 0, n_wins = 0, n_steps = 0;
    double return_sum = 0.0;
    for (int k = 0; k < k_steps; ++k) {
        if ((mode & MAZE_STEP_AUTORESET) && (st.flags & MAZE_ST_NEEDS_RESET)) {
            if ((mode & MAZE_STEP_WIN_NEXT) && (st.flags & MAZE_ST_WON)) {
                m += b.pool_stride;
                if (m >= b.num_mazes) m -= b.num_mazes;
                mz = load_maze(b, m);
            }
            bool wrapped;
            begin_episode(st, mz.start, __ldg(mz.tab + (mz.start & 0xffff) * mz.W + (mz.start >> 16)), wrapped);
            visit_bits_clear(b, e);
            if (wrapped)
                for (int i = 0; i < b.visit_slot; ++i) *VISIT_AT(b, e, i) = 0;
            reward = 0.0; term = 0; trunc = 0;
            ep_return = 0.0;
            target_changed = true;
        } else {
            const StepResult r = env_transition(b, e, st, mz, __ldcs(actions + (size_t)k * B + e) & 3, luts);
            reward = r.reward; term = r.term; trunc = r.trunc;
            ep_return += reward;
            ++n_steps;
            if (term | trunc) {
                ++n_episodes;
                n_wins += term;
                return_sum += ep_return;
            }
        }
        const size_t at = (size_t)k * B + e;
        if (tr.agent) __stcs(reinterpret_cast<int2*>(tr.agent) + at, make_int2(st.r, st.c));
        if (tr.best_dir)
            __stcs(reinterpret_cast<int2*>(tr.best_dir) + at,
                   best_dir_from_code((st.tab >> MAZE_TAB_CODE_SHIFT) & 7, st.r, st.c, mz.H, mz.W, mz.tor));
        if (tr.reward) __stcs(tr.reward + at, reward);
        if (tr.terminated) __stcs(tr.terminated + at, (uint8_t)term);
        if (tr.truncated) __stcs(tr.truncated + at, (uint8_t)trunc);
    }
    b.state[e] = pack_state(st);
    b.env_maze[e] = m;
    reinterpret_cast<int2*>(b.agent)[e] = make_int2(st.r, st.c);
    if (target_changed) {
        reinterpret_cast<int2*>(b.target)[e] = make_int2(mz.goal & 0xffff, mz.goal >> 16);
        if (b.target_dirty) *b.target_dirty = 1;
    }
    reinterpret_cast<int2*>(b.best_dir)[e] = best_dir_from_code((st.tab >> MAZE_TAB_CODE_SHIFT) & 7, st.r, st.c, mz.H, mz.W, mz.tor);
    b.reward[e] = reward;
    b.terminated[e] = (uint8_t)term;
    b.truncated[e] = (uint8_t)trunc;
    if (b.ep_return) b.ep_return[e] = ep_return;
    if (b.stats && n_steps) atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 3), n_steps);
    if (n_episodes) {
        if (b.stats) {
            atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 0), n_episodes);
            if (n_wins) atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 1), n_wins);
            if (n_episodes - n_wins) atomicAdd(reinterpret_cast<unsigned long long*>(b.stats + 2), n_episodes - n_wins);
        }
        if (b.ep_return && b.stats_return) atomicAdd(b.stats_return, return_sum);
    }
}

}  // namespace

extern "C" int maze_step_many(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, int k_steps, uint32_t mode,
                              const maze_step_trace* trace, int chunk_envs, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!actions) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_step_many: actions");
    if (k_steps < 1 || chunk_envs < 0) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_step_many: k_steps / chunk_envs");
    if (mode & MAZE_STEP_WIN_QUEUE)
        return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_step_many: MAZE_STEP_WIN_QUEUE needs a generation launch between steps; use maze_step");
    maze_step_trace tr = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (trace) tr = *trace;
    if (((uintptr_t)tr.agent & 7) || ((uintptr_t)tr.best_dir & 7) || ((uintptr_t)tr.reward & 7))
        return maze_fail_arg(ctx, MAZE_E_ALIGN, "maze_step_many: trace pointer alignment");
    // measured on B200 (tools/perf_step_many.py): one launch over all envs beats L2-sized chunks (the
    // locality that matters is each thread re-touching its own sectors within the burst), so chunking
    // is opt-in
    const int chunk = chunk_envs > 0 ? chunk_envs : b->num_envs;
    const StepLuts luts = step_luts(ctx);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int e0 = 0; e0 < b->num_envs; e0 += chunk) {
        const int e1 = e0 + chunk < b->num_envs ? e0 + chunk : b->num_envs;
        maze_step_many_kernel<<<(e1 - e0 + STEP_THREADS - 1) / STEP_THREADS, STEP_THREADS, 0, st>>>(*b, actions, k_steps, mode, luts, tr, e0, e1);
    }
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_step(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, uint32_t mode, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!actions) return maze_fail_arg(ctx, MAZE_E_NULL, "actions");
    if ((mode & MAZE_STEP_PACKED) && (!b->packed || ((uintptr_t)b->packed & 3)))
        return maze_fail_arg(ctx, MAZE_E_NULL, "maze_step: MAZE_STEP_PACKED needs batch.packed ([B] uint32)");
    if ((mode & MAZE_STEP_NO_WIDE) && !(mode & MAZE_STEP_PACKED))
        return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_step: MAZE_STEP_NO_WIDE without MAZE_STEP_PACKED would drop the step's outputs");
    const StepLuts luts = step_luts(ctx);
    const bool stats = b->ep_return || b->stats || ((mode & MAZE_STEP_WIN_QUEUE) && b->queue);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ept = b->num_envs < 64 * 1024 ? 1 : 2;   // small batches: more CTAs beats more loads per thread
    auto grid_for = [&](int e) { return (b->num_envs + STEP_THREADS * e - 1) / (STEP_THREADS * e); };
    const bool reverse = (ctx->step_launches++ & 1) != 0;
    auto launch = [&](auto kernel, int e) { kernel<<<grid_for(e), STEP_THREADS, 0, st>>>(*b, actions, mode, luts, reverse); };
#define MAZE_STEP_DISPATCH(EPT_)                                                                          \
    do {                                                                                                  \
        if (stats) { if (tiled) launch(maze_step_kernel<EPT_, true, true>, EPT_); else launch(maze_step_kernel<EPT_, true, false>, EPT_); } \
        else       { if (tiled) launch(maze_step_kernel<EPT_, false, true>, EPT_); else launch(maze_step_kernel<EPT_, false, false>, EPT_); } \
    } while (0)
    const bool tiled = b->visit_tiled != 0;
    if (ept == 2) MAZE_STEP_DISPATCH(2);
    else MAZE_STEP_DISPATCH(1);
#undef MAZE_STEP_DISPATCH
    MAZE_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int maze_reset(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* mask, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    const int grid = (b->num_envs + STEP_THREADS - 1) / STEP_THREADS;
    maze_reset_kernel<<<grid, STEP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*b, mask);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}
