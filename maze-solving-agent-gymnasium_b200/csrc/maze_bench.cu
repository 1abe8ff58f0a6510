// Micro-benchmark of the access pattern that bounds maze_step (DESIGN.md section 4.1): per launch, every env streams
// its coalesced words (13 B read, 34 + 8 B written = the step kernel's 47 B of streams plus the 8-byte state store)
// and a fraction of the envs do ONE 2-byte read-modify-write at a scattered address of a large array (the visit
// counter of the block stepped onto).  No maze logic: what remains is what HBM3e + L2 give this pattern.
//   pattern 0  uniform random element of the array
//   pattern 1  cell-major [slot, B] addressing: element = cell * B + env with a random cell per env and launch
//              (neighbouring envs land in different 64-byte atoms, like decorrelated agents)
//   pattern 2  as 1, but the 32 envs of a warp share the cell (agents that still walk together: one atom per warp)
// Pattern 1 can also model the lag-1 re-touches of a random walk: of the envs that did an RMW in the previous launch,
// retouch_per_1024 of every 1024 go back to that launch's cell instead of drawing a new one.  `order` 1 runs the CTAs
// in reverse on odd launches (maze_step's order), so that the envs stepped last in one launch are stepped first in the
// next.  `hints` picks the L2 cache policies of the state / env_maze words and of the array element:
//   0  no hint (plain loads and stores)
//   1  state, env_maze and array element all evict_last
//   2  state and env_maze evict_first, array element evict_last
//   3  state and env_maze evict_last, array element no hint
#include "maze_env.cuh"

namespace {

__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}

__device__ __forceinline__ uint64_t l2_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__global__ void __launch_bounds__(256)
bench_scatter_kernel(const uint64_t* __restrict__ state_in, uint64_t* __restrict__ state_out, const int32_t* __restrict__ env_maze,
                     const uint8_t* __restrict__ actions, int2* __restrict__ agent, int2* __restrict__ best_dir, double* __restrict__ reward,
                     uint8_t* __restrict__ term, uint8_t* __restrict__ trunc, uint16_t* __restrict__ arr, long long n_elems, int B, int slot,
                     int pattern, uint32_t rmw_per_1024, uint32_t launch, int streams, int order, uint32_t retouch_per_1024, int hints) {
    const int blk = (order && (launch & 1)) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
    const int e = blk * 256 + threadIdx.x;
    if (e >= B) return;
    const bool hint_s = hints != 0, hint_a = hints == 1 || hints == 2;
    const uint64_t pol_s = hints == 2 ? l2_evict_first() : l2_policy(), pol_a = l2_policy();
    uint64_t s = 0;
    int m = 0, a = 0;
    if (streams) {
        s = hint_s ? pol_load(reinterpret_cast<const unsigned long long*>(state_in) + e, pol_s) : state_in[e];
        m = hint_s ? pol_load(env_maze + e, pol_s) : env_maze[e];
        a = __ldcs(actions + e);
    }
    auto hash_at = [&](uint32_t l) { return mix32((uint32_t)e * 0x9E3779B9u + l * 0x85EBCA6Bu); };
    const uint32_t h = hash_at(launch);
    uint32_t v = 0;
    if ((h & 1023u) < rmw_per_1024) {
        long long idx;
        if (pattern == 0) {
            idx = (long long)(((unsigned long long)mix32(h + 1) << 32 | mix32(h + 2)) % (unsigned long long)n_elems);
        } else if (pattern == 2) {
            idx = (long long)(mix32(((uint32_t)e >> 5) * 0x9E3779B9u + launch) % (uint32_t)slot) * B + e;
        } else {
            // the cell of launch l is the cell of launch l - 1 while l re-touches (bounded walk back: chains of 8 are rare)
            uint32_t hl = h;
            for (uint32_t l = launch, n = 0; l > 0 && n < 8; --l, ++n) {
                const uint32_t hp = hash_at(l - 1);
                if ((hp & 1023u) >= rmw_per_1024 || (mix32(hl + 4) & 1023u) >= retouch_per_1024) break;
                hl = hp;
            }
            idx = (long long)(mix32(hl + 3) % (uint32_t)slot) * B + e;
        }
        uint16_t* p = arr + idx;
        v = hint_a ? pol_load(p, pol_a) : *p;
        const unsigned nv = (uint16_t)(v + 1 + (uint32_t)(s & 1));
        if (hint_a) pol_store(p, nv, pol_a);
        else *p = (uint16_t)nv;
    }
    if (streams) {
        const unsigned long long ns = s + v + (uint64_t)(m + a);
        if (hint_s) pol_store(reinterpret_cast<unsigned long long*>(state_out) + e, ns, pol_s);
        else state_out[e] = ns;
        __stcs(agent + e, make_int2((int)(s & 0xff), (int)((s >> 8) & 0xff)));
        __stcs(best_dir + e, make_int2(a, m));
        __stcs(reward + e, (double)v);
        __stcs(term + e, (uint8_t)(v & 1));
        __stcs(trunc + e, (uint8_t)0);
    }
}

}  // namespace

// arr: uint16 [n_elems] (n_elems >= slot * B for patterns 1, 2).  rmw_per_1024: envs out of 1024 that touch the array
// per launch (the step kernel: ~410).  streams != 0 adds the coalesced reads / writes of maze_step.
extern "C" int maze_bench_scatter_rmw(maze_ctx* ctx, const maze_env_batch* b, const uint8_t* actions, uint16_t* arr, int64_t n_elems, int pattern,
                                      int rmw_per_1024, uint32_t launch, int streams, int order, int retouch_per_1024, int hints, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (int rc = maze_check_batch(ctx, b)) return rc;
    if (!arr || !actions || n_elems < 1 || pattern < 0 || pattern > 2 || order < 0 || order > 1 || retouch_per_1024 < 0 || hints < 0 || hints > 3)
        return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_bench_scatter_rmw arguments");
    if (pattern != 0 && n_elems < (int64_t)b->slot * b->num_envs) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_bench_scatter_rmw: array smaller than slot * B");
    bench_scatter_kernel<<<(b->num_envs + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        b->state, b->state, b->env_maze, actions, reinterpret_cast<int2*>(b->agent), reinterpret_cast<int2*>(b->best_dir), b->reward, b->terminated,
        b->truncated, arr, (long long)n_elems, b->num_envs, b->slot, pattern, (uint32_t)rmw_per_1024, launch, streams, order,
        (uint32_t)retouch_per_1024, hints);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}
