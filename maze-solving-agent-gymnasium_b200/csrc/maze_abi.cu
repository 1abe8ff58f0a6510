// Context management and host-side helpers of the C ABI.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include "maze_common.cuh"

int maze_fail_cuda(maze_ctx* ctx, cudaError_t e, const char* what) {
    if (ctx) snprintf(ctx->err, sizeof(ctx->err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return (int)e;
}

int maze_fail_arg(maze_ctx* ctx, int code, const char* what) {
    if (ctx) snprintf(ctx->err, sizeof(ctx->err), "argument error %d: %s", code, what);
    return code;
}

// argument validation shared by every entry point that takes a maze_env_batch
int maze_check_batch(maze_ctx* ctx, const maze_env_batch* b) {
    if (!b) return maze_fail_arg(ctx, MAZE_E_NULL, "batch");
    if (!b->meta || !b->table || !b->env_maze || !b->state || !b->visits || !b->agent || !b->target ||
        !b->best_dir || !b->reward || !b->terminated || !b->truncated)
        return maze_fail_arg(ctx, MAZE_E_NULL, "batch pointer");
    if (b->num_envs <= 0 || b->num_mazes <= 0 || b->slot <= 0 || (b->slot & 1))
        return maze_fail_arg(ctx, MAZE_E_RANGE, "num_envs / num_mazes / slot (must be even)");
    if (b->visit_slot < b->slot || (b->visit_tiled != 0 && b->visit_tiled != 1))
        return maze_fail_arg(ctx, MAZE_E_RANGE, "visit_slot (>= slot) / visit_tiled (0 or 1)");
    if (b->visit_bits && (b->visit_bits_pitch < 1 || b->visit_bits_stride < b->visit_bits_pitch || (b->visit_bits_stride & 3) ||
                          ((uintptr_t)b->visit_bits & 15)))
        return maze_fail_arg(ctx, MAZE_E_RANGE, "visit_bits: pitch >= 1, stride a multiple of 4 words, 16-byte aligned");
    if (b->visit_cell_stride <= 0 || b->visit_env_stride <= 0)
        return maze_fail_arg(ctx, MAZE_E_RANGE, "visit strides (cell-major: B, 1; env-major: 1, slot)");
    if (((uintptr_t)b->meta & 15) || ((uintptr_t)b->state & 7) || ((uintptr_t)b->agent & 7) ||
        ((uintptr_t)b->target & 7) || ((uintptr_t)b->best_dir & 7) || ((uintptr_t)b->reward & 7) ||
        ((uintptr_t)b->visits & 3))
        return maze_fail_arg(ctx, MAZE_E_ALIGN, "batch pointer alignment");
    return 0;
}


extern "C" int maze_abi_version(void) { return MAZE_ABI_VERSION; }

extern "C" int maze_sizeof(int which) {
    switch (which) {
        case 0: return (int)sizeof(maze_env_batch);
        case 1: return (int)sizeof(maze_q_agent);
        case 2: return (int)sizeof(maze_replay);
        case 3: return (int)sizeof(maze_step_trace);
        case 4: return (int)sizeof(maze_dqn_net);
        default: return -1;
    }
}

extern "C" int maze_ctx_create(maze_ctx** out, int device) {
    if (!out) return MAZE_E_NULL;
    *out = nullptr;
    maze_ctx* ctx = new (std::nothrow) maze_ctx();
    if (!ctx) return MAZE_E_RANGE;
    memset(ctx, 0, sizeof(*ctx));
    ctx->device = device;
    // Same libm `exp` the reference's math.exp calls (base_maze_env.py:194,200), same
    // expression order, so the tables are bit-identical to what the reference computes.
    for (int i = 0; i < 256; ++i) {
        ctx->h_lut_revisit[i] = 0.0 - (1 - std::exp(-0.2 * i));
        ctx->h_lut_invalid[i] = 0.0 - (1 - std::exp(-0.15 * i));
    }
    ctx->h_shaping[0] = 0 * 0.5 - 0.05;    // base_maze_env.py:192
    ctx->h_shaping[1] = 1 * 0.5 - 0.05;
    ctx->h_shaping[2] = 0.0;               // unused (|delta| <= 1)
    ctx->h_shaping[3] = -1 * 0.5 - 0.05;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_lut_revisit, 256 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_lut_invalid, 256 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_counter, 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_lut_revisit, ctx->h_lut_revisit, 256 * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_lut_invalid, ctx->h_lut_invalid, 256 * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) {
        int rc = (int)e;
        cudaFree(ctx->d_lut_revisit);
        cudaFree(ctx->d_lut_invalid);
        cudaFree(ctx->d_counter);
        delete ctx;
        return rc;
    }
    *out = ctx;
    return 0;
}

extern "C" void maze_ctx_destroy(maze_ctx* ctx) {
    if (!ctx) return;
    cudaFree(ctx->d_lut_revisit);
    cudaFree(ctx->d_lut_invalid);
    cudaFree(ctx->d_counter);
    cudaFree(ctx->d_scratch);
    maze_net_profile_free(ctx);
    delete ctx;
}

extern "C" const char* maze_last_error(maze_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }

// Host-only: usable without a GPU (the tables are plain libm arithmetic).
extern "C" int maze_reward_lut(maze_ctx* ctx, int kind, double* out) {
    if (!out) return MAZE_E_NULL;
    double rev[256], inv[256];
    for (int i = 0; i < 256; ++i) {
        rev[i] = 0.0 - (1 - std::exp(-0.2 * i));
        inv[i] = 0.0 - (1 - std::exp(-0.15 * i));
    }
    memset(out, 0, 256 * sizeof(double));
    if (kind == 0) memcpy(out, rev, sizeof(rev));
    else if (kind == 1) memcpy(out, inv, sizeof(inv));
    else if (kind == 2) { out[0] = -1 * 0.5 - 0.05; out[1] = 0 * 0.5 - 0.05; out[2] = 1 * 0.5 - 0.05; }
    else return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_reward_lut kind");
    return 0;
}

// Host-only: packed step records -> the wide arrays (see MAZE_STEP_PACKED in the header).
extern "C" int maze_step_decode_host(const uint32_t* records, int64_t n, const int32_t* shape, const uint8_t* toroidal, int32_t* agent,
                                     int32_t* best_dir, double* reward, uint8_t* terminated, uint8_t* truncated) {
    if (!records || n < 0) return MAZE_E_NULL;
    double lut[4][256];
    memset(lut, 0, sizeof(lut));
    for (int i = 0; i < 256; ++i) {
        lut[MAZE_REC_KIND_REVISIT][i] = 0.0 - (1 - std::exp(-0.2 * i));
        lut[MAZE_REC_KIND_INVALID][i] = 0.0 - (1 - std::exp(-0.15 * i));
    }
    lut[MAZE_REC_KIND_SHAPING][0] = -1 * 0.5 - 0.05;
    lut[MAZE_REC_KIND_SHAPING][1] = 0 * 0.5 - 0.05;
    lut[MAZE_REC_KIND_SHAPING][2] = 1 * 0.5 - 0.05;
    lut[MAZE_REC_KIND_CONST][MAZE_REC_CONST_ONE] = 1.0;
    lut[MAZE_REC_KIND_CONST][MAZE_REC_CONST_MINUS_ONE] = -1.0;
    for (int64_t e = 0; e < n; ++e) {
        const uint32_t rec = records[e];
        const int r = (int)(rec & 0xff), c = (int)((rec >> 8) & 0xff), code = (int)((rec >> MAZE_REC_CODE_SHIFT) & 7);
        if (agent) { agent[2 * e] = r; agent[2 * e + 1] = c; }
        if (best_dir) {
            int br = 0, bc = 0;
            if (code < 4) {
                const int dr = (code == 0) - (code == 1), dc = (code == 2) - (code == 3);
                int nr = r + dr, nc = c + dc;
                if (toroidal && toroidal[e] && shape) {
                    const int H = shape[2 * e], W = shape[2 * e + 1];
                    nr = nr < 0 ? H - 1 : (nr >= H ? 0 : nr);
                    nc = nc < 0 ? W - 1 : (nc >= W ? 0 : nc);
                }
                br = r - nr;
                bc = c - nc;
            }
            best_dir[2 * e] = br;
            best_dir[2 * e + 1] = bc;
        }
        if (reward) reward[e] = lut[(rec >> MAZE_REC_KIND_SHIFT) & 3][(rec >> MAZE_REC_INDEX_SHIFT) & 0xff];
        if (terminated) terminated[e] = (uint8_t)((rec >> MAZE_REC_TERM_SHIFT) & 1);
        if (truncated) truncated[e] = (uint8_t)((rec >> MAZE_REC_TRUNC_SHIFT) & 1);
    }
    return 0;
}
