// Per-env transition pieces shared by the step kernel and the fused Q-learning rollout (sm_100a).
// Reference semantics: gymnasium_env/envs/base_maze_env.py:136-210, lib/maze_view.py:165-197.
#pragma once
#include "maze_common.cuh"

struct StepLuts {
    const double* revisit;  // [256]
    const double* invalid;  // [256]
    double shaping_same, shaping_closer, shaping_farther;   // D[prev]-D[cur] = 0, +1, -1
};

inline StepLuts step_luts(const maze_ctx* ctx) {
    StepLuts l;
    l.revisit = ctx->d_lut_revisit;
    l.invalid = ctx->d_lut_invalid;
    l.shaping_same = ctx->h_shaping[0];
    l.shaping_closer = ctx->h_shaping[1];
    l.shaping_farther = ctx->h_shaping[3];
    return l;
}

// Visit counters are stored cell-major: entry (cell idx, env e) at idx * num_envs + e.  Envs that
// share a maze are contiguous and start from the same block, so lanes of a warp standing on the
// same block hit the same 64 bytes; lanes on different blocks cost one DRAM line each, exactly
// like an env-major layout would.
#define VISIT_AT(b, e, idx) ((b).visits + (size_t)(idx) * (b).visit_cell_stride + (size_t)(e) * (b).visit_env_stride)

// ---- cache-policy helpers --------------------------------------------------------------------
// What one step touches per env, and how long it is worth keeping in the 126 MB L2:
//   state word, maze id (12 B)   re-read by the next step
//   step table (6.5 KB / maze)   shared by every env of the maze
//   visit counter (2 B RMW)      54 GB array, random access
//   action, obs, reward, flags   written / read once               -> always streaming (.cs)
// The first three are all loaded and stored L2 evict_last.  The default policy and evict_first
// measured within 2 % of it on B200, except evict_first on the visit sectors, which was 20 %
// slower: the store misses the sector its own load fetched (DESIGN.md §4.1).  With maze_step's CTA order
// reversed on every other launch, evict_first on state / env_maze and no hint on the visits were 1 % and
// 2.7 % slower than evict_last.
__device__ __forceinline__ uint64_t l2_policy() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long pol_load(const unsigned long long* p, uint64_t pol) {
    unsigned long long v;
    asm volatile("ld.global.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int pol_load(const int* p, uint64_t pol) {
    int v;
    asm volatile("ld.global.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ unsigned pol_load(const uint16_t* p, uint64_t pol) {
    unsigned short v;
    asm volatile("ld.global.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int pol_load_nc(const uint8_t* p, uint64_t pol) {   // read-only data
    unsigned v;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return (int)v;
}
__device__ __forceinline__ void pol_store(unsigned long long* p, unsigned long long v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void pol_store(int* p, int v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.s32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void pol_store(uint16_t* p, unsigned v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.u16 [%0], %1, %2;" ::"l"(p), "h"((unsigned short)v), "l"(pol) : "memory");
}

// index of block (r, c) in an env's visit array (see maze_env_batch.visit_tiled)
__device__ __forceinline__ int visit_index(const maze_env_batch& b, int r, int c, int W) {
    if (b.visit_tiled) return (((r >> 2) * ((W + 3) >> 2) + (c >> 2)) << 4) | ((r & 3) << 2) | (c & 3);
    return r * W + c;
}

// "Visited in this episode" bitmap (maze_env_batch.visit_bits; optional).
__device__ __forceinline__ void visit_bit_set(const maze_env_batch& b, int e, int r, int c) {
    if (b.visit_bits) atomicOr(b.visit_bits + (size_t)e * b.visit_bits_stride + r * b.visit_bits_pitch + (c >> 5), 1u << (c & 31));
}
__device__ __forceinline__ void visit_bits_clear(const maze_env_batch& b, int e) {   // an episode starts
    if (!b.visit_bits) return;
    uint4* p = reinterpret_cast<uint4*>(b.visit_bits + (size_t)e * b.visit_bits_stride);
    for (int i = 0; i < (b.visit_bits_stride >> 2); ++i) p[i] = make_uint4(0, 0, 0, 0);
}

// Zero the visit counters of the lanes in `need` (epoch wrap-around: once per 255 episodes per
// env; envs sharing a maze wrap together, so the lanes of a warp usually clear side by side).
// Must be called by all 32 lanes.
__device__ __forceinline__ void warp_clear_visits(unsigned need, const maze_env_batch& b, int e) {
    if (need & (1u << (threadIdx.x & 31)))
        for (int i = 0; i < b.visit_slot; ++i) *VISIT_AT(b, e, i) = 0;
}

// Episode (re)start: BaseMazeEnv.reset, base_maze_env.py:136-161.  The start block is NOT
// marked visited (:159), only excluded from non_visited (:149).
__device__ __forceinline__ void begin_episode(EnvState& s, int start, int tab_at_start, bool& wrapped) {
    s.r = start & 0xffff;
    s.c = start >> 16;
    s.consec = 0;
    s.flags = 0;
    s.steps = 0;
    s.epoch += 1;
    wrapped = s.epoch > 255;
    if (wrapped) s.epoch = 1;
    s.tab = tab_at_start;
}

// What a kernel needs to know about one maze (32-byte meta record, L1/L2 resident).
struct MazeView {
    int H, W, start, goal, max_steps;
    bool tor;
    const uint8_t* tab;
};

__device__ __forceinline__ MazeView load_maze(const maze_env_batch& b, int m) {
    const int4* mp = reinterpret_cast<const int4*>(b.meta + (size_t)m * MAZE_META_WORDS);
    const int4 m0 = __ldg(mp), m1 = __ldg(mp + 1);
    MazeView v;
    v.H = m0.x; v.W = m0.y; v.start = m0.z; v.goal = m0.w;
    v.max_steps = m1.x;
    v.tor = (m1.y & MAZE_FLAG_TOROIDAL) != 0;
    v.tab = b.table + (size_t)m * b.slot;
    return v;
}

struct StepResult {
    double reward;
    int term, trunc;
};

// One BaseMazeEnv.step for env e (no autoreset handling; the caller owns NEEDS_RESET).  The same
// rules as maze_step_kernel, written for one env at a time (used inside multi-step loops).
__device__ __forceinline__ StepResult env_transition(const maze_env_batch& b, int e, EnvState& st, const MazeView& mz,
                                                     int a, const StepLuts& luts) {
    StepResult out = {0.0, 0, 0};
    int dr, dc;
    action_delta(a, dr, dc);
    int nr = st.r + dr, nc = st.c + dc;
    bool inb = true;
    if (mz.tor) {   // lib/maze_view.py:185-186
        nr = nr < 0 ? mz.H - 1 : (nr >= mz.H ? 0 : nr);
        nc = nc < 0 ? mz.W - 1 : (nc >= mz.W ? 0 : nc);
    } else {        // lib/maze_view.py:169
        inb = (nr > 0) & (nr < mz.H - 1) & (nc > 0) & (nc < mz.W - 1);
    }
    const int idx = nr * mz.W + nc;
    const int tb = inb ? __ldg(mz.tab + idx) : 0;
    if (inb && (tb & MAZE_TAB_OPEN)) {
        const uint64_t pol = l2_policy();
        uint16_t* vp = VISIT_AT(b, e, visit_index(b, nr, nc, mz.W));
        const unsigned vis = pol_load(vp, pol);
        const int cnt = ((int)(vis >> 8) == st.epoch) ? (int)(vis & 0xff) : 0;
        if (cnt == 0) {
            if ((nr | (nc << 16)) == mz.goal) {
                out.reward = 1.0;   // base_maze_env.py:185-187
                out.term = 1;
            } else {                // :189-192
                const int dd = ((st.tab >> MAZE_TAB_D4_SHIFT) - (tb >> MAZE_TAB_D4_SHIFT)) & 3;
                out.reward = dd == 1 ? luts.shaping_closer : (dd == 3 ? luts.shaping_farther : luts.shaping_same);
            }
        } else {
            out.reward = __ldg(luts.revisit + cnt);   // :194
        }
        pol_store(vp, (unsigned)((st.epoch << 8) | (cnt < 255 ? cnt + 1 : 255)), pol);   // :196
        visit_bit_set(b, e, nr, nc);
        st.r = nr;
        st.c = nc;
        st.tab = tb;
        st.consec = 0;
        int nm = (st.flags >> MAZE_ST_NMOVES_SHIFT) & 3;
        nm = nm < 2 ? nm + 1 : 2;
        st.flags = (a << MAZE_ST_MOVE_SHIFT) | (nm << MAZE_ST_NMOVES_SHIFT);
    } else {
        st.consec = st.consec < 255 ? st.consec + 1 : 255;   // :199-200
        out.reward = __ldg(luts.invalid + st.consec);
        st.flags &= ~(MAZE_ST_NEEDS_RESET | MAZE_ST_WON);
    }
    st.steps = st.steps < 65535 ? st.steps + 1 : 65535;
    if (st.steps > mz.max_steps) {   // :205-208 (overrides a goal reward on the same step)
        out.trunc = 1;
        out.reward = -1.0;
    }
    if (out.term | out.trunc) st.flags |= MAZE_ST_NEEDS_RESET | (out.term ? MAZE_ST_WON : 0);
    return out;
}
