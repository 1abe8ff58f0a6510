// Shared device helpers for the maze kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "maze_b200.h"

#define MAZE_CHECK(call)                                                          \
    do {                                                                          \
        cudaError_t _e = (call);                                                  \
        if (_e != cudaSuccess) return maze_fail_cuda(ctx, _e, #call);             \
    } while (0)

struct maze_ctx {
    int device;
    double* d_lut_revisit;   // [256]
    double* d_lut_invalid;   // [256]
    int*    d_counter;       // [4] work-distribution counters (zeroed before each use)
    double h_lut_revisit[256];
    double h_lut_invalid[256];
    double h_shaping[4];     // index = (D[prev]-D[cur]) & 3 : 0 -> 0, 1 -> +1, 3 -> -1
    int    num_sms;
    void*  d_scratch;       // library-owned scratch (candidate wall planes of scored generation), grown on demand
    size_t scratch_bytes;
    void*  net_profile;     // maze_net.cu: in-situ launch timing (events), created on first use
    unsigned step_launches; // maze_step calls so far: odd ones run the CTAs in reverse order
    char   err[512];
};

void maze_net_profile_free(maze_ctx* ctx);   // maze_net.cu
int maze_fail_cuda(maze_ctx* ctx, cudaError_t e, const char* what);
int maze_fail_arg(maze_ctx* ctx, int code, const char* what);
int maze_check_batch(maze_ctx* ctx, const maze_env_batch* b);

// ---------------------------------------------------------------------------------------------
// packed per-env state (see include/maze_b200.h)
struct EnvState {
    int r, c, consec, flags, steps, epoch, tab;
};

__device__ __forceinline__ EnvState unpack_state(uint64_t s) {
    EnvState e;
    e.r = (int)(s & 0xff);
    e.c = (int)((s >> 8) & 0xff);
    e.consec = (int)((s >> 16) & 0xff);
    e.flags = (int)((s >> 24) & 0xff);
    e.steps = (int)((s >> 32) & 0xffff);
    e.epoch = (int)((s >> 48) & 0xff);
    e.tab = (int)((s >> 56) & 0xff);
    return e;
}

__device__ __forceinline__ uint64_t pack_state(const EnvState& e) {
    uint32_t lo = (uint32_t)e.r | ((uint32_t)e.c << 8) | ((uint32_t)e.consec << 16) | ((uint32_t)e.flags << 24);
    uint32_t hi = (uint32_t)e.steps | ((uint32_t)e.epoch << 16) | ((uint32_t)e.tab << 24);
    return (uint64_t)lo | ((uint64_t)hi << 32);
}

// action -> (dr, dc): 0 down, 1 up, 2 right, 3 left   (base_maze_env.py:19-24)
__device__ __forceinline__ void action_delta(int a, int& dr, int& dc) {
    dr = (a == 0) - (a == 1);
    dc = (a == 2) - (a == 3);
}

// `agent - best_next` from the 3-bit code stored in the step table (base_maze_env.py:122).
// On the torus best_next is wrapped (toroidal_maze_env.py:79-81), giving +-(S-1) components.
__device__ __forceinline__ int2 best_dir_from_code(int code, int r, int c, int H, int W, bool tor) {
    if (code >= 4) return make_int2(0, 0);
    int dr, dc;
    action_delta(code, dr, dc);
    int nr = r + dr, nc = c + dc;
    if (tor) {
        nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
        nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
    }
    return make_int2(r - nr, c - nc);
}

// streaming (evict-first) stores for outputs nobody re-reads on the device
__device__ __forceinline__ void st_cs(int2* p, int2 v) { __stcs(p, v); }
__device__ __forceinline__ void st_cs(double* p, double v) { __stcs(p, v); }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG: stream = (seed, sequence id), 4 x 32 bits per call.
struct Philox {
    uint32_t k0, k1;
    uint32_t c0, c1, c2, c3;
    uint32_t o0, o1, o2, o3;
    int have;

    // `sub` selects one of 2^32 sub-streams of (seed, seq) (each 2^32 blocks long)
    __host__ __device__ void init(uint64_t seed, uint64_t seq, uint32_t sub = 0) {
        k0 = (uint32_t)seed;
        k1 = (uint32_t)(seed >> 32);
        c0 = 0; c1 = sub;
        c2 = (uint32_t)seq;
        c3 = (uint32_t)(seq >> 32);
        have = 0;
    }
    __host__ __device__ static inline void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
        uint64_t p = (uint64_t)a * b;
        hi = (uint32_t)(p >> 32);
        lo = (uint32_t)p;
    }
    __host__ __device__ void refill() {
        uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = c3, a = k0, b = k1;
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            uint32_t hi0, lo0, hi1, lo1;
            mulhilo(0xD2511F53u, x0, hi0, lo0);
            mulhilo(0xCD9E8D57u, x2, hi1, lo1);
            uint32_t y0 = hi1 ^ x1 ^ a, y1 = lo1, y2 = hi0 ^ x3 ^ b, y3 = lo0;
            x0 = y0; x1 = y1; x2 = y2; x3 = y3;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        o0 = x0; o1 = x1; o2 = x2; o3 = x3;
        if (++c0 == 0) ++c1;
        have = 4;
    }
    __host__ __device__ uint32_t next() {
        if (have == 0) refill();
        const uint32_t v = o0;
        o0 = o1; o1 = o2; o2 = o3;
        --have;
        return v;
    }
    // uniform integer in [0, n) (multiply-shift; bias < n / 2^32)
    __host__ __device__ uint32_t below(uint32_t n) {
        return (uint32_t)(((uint64_t)next() * n) >> 32);
    }
};
