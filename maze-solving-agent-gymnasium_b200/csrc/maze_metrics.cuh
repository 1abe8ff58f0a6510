// Difficulty metrics of one bordered perfect maze held in shared memory (one CTA per maze).
//
// McClendon complexity / difficulty (maze_complexity_evaluation.py:38-329) and Kim-Crawfis
// L / D / DE (metrics_calculator.py:11-26,71-173), restated on the maze's spanning tree rooted at
// `start` (see oracle/metrics.py, which is the specification):
//   - the reference's graph G is the maze tree compressed onto its nodes (start, dead ends,
//     corners, >2-neighbour cells); every node is a logical cell, so all arrays are per cell
//   - hallways >= 1 are the components of (plain nodes) with their adjacent 3-way junctions;
//     each tree edge contributes (d, 1/(2d)) to at most one hallway; branch = the solution
//     junction run / hanging subtree the component is attached to
//   - difficulty = ln(C0 * prod_b (C_b + 1)), complexity = ln(C0 + sum_b C_b)
// Input: f.grid (0 wall / !=0 open, goal marked 2) and f.dist = BFS distances from start.
#pragma once
#include "maze_fields.cuh"

struct MetricsSmem {
    unsigned short* pnode;    // [cells] parent node (cell index), 0xffff for start
    unsigned short* dpar;     // [cells] blocks strictly between node and parent node
    unsigned short* comp;     // [cells] component root of a plain node
    unsigned short* minleaf;  // [cells] smallest off-solution dead-end rank in the subtree
    uint8_t* flags;           // [cells]
    unsigned int* dsum;       // [cells] sum of d over the hallway of component root
    double* ssum;             // [cells] sum of 1/(2d)
    double* bsum;             // [cells] branch complexity by branch key
};

constexpr int MF_NB = 0x07, MF_TURN = 0x08, MF_SOL = 0x10, MF_NODE = 0x20, MF_PDIR_SHIFT = 6;   // bits 6-7: parent direction

// The four u16 arrays (8 bytes per cell) live in the BFS queue of FieldSmem, which is dead once
// the distances from start exist (2 * H * W bytes > 8 * cells); the rest is carved from `base`.
__host__ __device__ inline size_t metrics_smem_bytes(int cells) {
    auto up = [](size_t x) { return (x + 15) & ~(size_t)15; };
    return 2 * up(8 * (size_t)cells) + up(4 * (size_t)cells) + up((size_t)cells);
}

__device__ inline MetricsSmem metrics_smem_carve(unsigned char* base, int cells, unsigned short* bfs_queue) {
    auto up = [](size_t x) { return (x + 15) & ~(size_t)15; };
    MetricsSmem m;
    size_t o = 0;
    m.ssum = reinterpret_cast<double*>(base + o); o += up(8 * (size_t)cells);
    m.bsum = reinterpret_cast<double*>(base + o); o += up(8 * (size_t)cells);
    m.dsum = reinterpret_cast<unsigned int*>(base + o); o += up(4 * (size_t)cells);
    m.flags = base + o;
    m.pnode = bfs_queue;
    m.dpar = bfs_queue + cells;
    m.comp = bfs_queue + 2 * cells;
    m.minleaf = bfs_queue + 3 * cells;
    return m;
}

// 16-bit atomic min on shared memory (two cells share a 32-bit word); true if v was stored, false if the
// cell already held something <= v
__device__ __forceinline__ bool atomic_min_u16(unsigned short* p, unsigned short v) {
    unsigned int* w = reinterpret_cast<unsigned int*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
    const bool hi = (reinterpret_cast<uintptr_t>(p) & 2) != 0;
    unsigned int old = *w;
    for (;;) {
        const unsigned short cur = hi ? (unsigned short)(old >> 16) : (unsigned short)(old & 0xffffu);
        if (cur <= v) return false;
        const unsigned int repl = hi ? ((old & 0x0000ffffu) | ((unsigned int)v << 16)) : ((old & 0xffff0000u) | v);
        const unsigned int seen = atomicCAS(w, old, repl);
        if (seen == old) return true;
        old = seen;
    }
}

struct MazeMetrics {
    double difficulty, complexity, L, DE, D;
    int sol_len, de_count;
    double ext[MAZE_METRIC_EXT_WORDS];   // filled when maze_metrics(..., ext = true); see include/maze_b200.h
};

// All threads of the CTA call this; the result is valid on thread 0.
// with_kc = false skips the (sequential) Kim-Crawfis DE pass: DE / de_count are then 0.
// ext = true (needs with_kc) also fills out.ext with the metrics the reference defines but never calls
// (metrics_calculator.py:18-69,175-244), bit-identical: same divisions, sums in row-major dead-end order.
__device__ inline void maze_metrics(const FieldSmem& f, const MetricsSmem& ms, int Hb, int Wb,
                                    int start_idx, int goal_idx, MazeMetrics& out, bool with_kc = true, bool ext = false) {
    __shared__ double s_D0, s_S0, s_red[2][METRIC_THREADS / 32];
    __shared__ int s_dcount, s_sol_counts[3], s_open, s_de_counts[3];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int nr = (Hb - 1) / 2, nc = (Wb - 1) / 2, cells = nr * nc;
    auto cell_block = [&](int ci) { return (2 * (ci / nc) + 1) * Wb + 2 * (ci % nc) + 1; };
    auto block_cell = [&](int bi) { return ((bi / Wb) >> 1) * nc + ((bi % Wb) >> 1); };
    const int offs[4] = {-Wb, Wb, -1, 1};
    const int start_c = block_cell(start_idx), goal_c = block_cell(goal_idx);
    if (f.dist[goal_idx] == DIST_INF) {   // goal not reachable from start: not a maze the reference can score
        if (tid == 0) {
            out.difficulty = out.complexity = out.L = out.DE = out.D = nan("");
            out.sol_len = 0;
            out.de_count = 0;
            if (ext)
                for (int i = 0; i < MAZE_METRIC_EXT_WORDS; ++i) out.ext[i] = nan("");
        }
        __syncthreads();
        return;
    }
    const int sol_len = (int)f.dist[goal_idx] + 1;

    // ---- 1. per-cell neighbour count / turn / node flags
    for (int ci = tid; ci < cells; ci += nthr) {
        const int b = cell_block(ci);
        const int up = f.grid[b - Wb] != 0, dn = f.grid[b + Wb] != 0, lf = f.grid[b - 1] != 0, rt = f.grid[b + 1] != 0;
        const int nb = up + dn + lf + rt;
        const int turn = (nb == 2) && !((up && dn) || (lf && rt));
        const int d = f.dist[b];
        const int node = ((nb != 2) || turn || ci == start_c) && d != DIST_INF;   // unreachable cells play no part
        // direction of the tree parent (the open neighbour one block closer to start; the last match in the
        // order up, down, left, right, as the sequential walks used to pick it), kept in the two top flag bits
        int pdir = 0;
        if (up && (int)f.dist[b - Wb] == d - 1) pdir = 0;
        if (dn && (int)f.dist[b + Wb] == d - 1) pdir = 1;
        if (lf && (int)f.dist[b - 1] == d - 1) pdir = 2;
        if (rt && (int)f.dist[b + 1] == d - 1) pdir = 3;
        ms.flags[ci] = (uint8_t)(nb | (turn ? MF_TURN : 0) | (node ? MF_NODE : 0) | (pdir << MF_PDIR_SHIFT));
        ms.dsum[ci] = 0u;
        ms.ssum[ci] = 0.0;
        ms.bsum[ci] = 0.0;
        ms.minleaf[ci] = 0xffffu;
        ms.comp[ci] = 0xffffu;
        ms.pnode[ci] = 0xffffu;
        ms.dpar[ci] = 0;
    }
    if (tid == 0) { s_D0 = 0.0; s_S0 = 0.0; s_dcount = 0; s_open = 0; s_de_counts[0] = s_de_counts[1] = s_de_counts[2] = 0; }
    __syncthreads();
    if (ext) {   // calculate_density :18-20
        int open = 0;
        for (int i = tid; i < Hb * Wb; i += nthr) open += f.grid[i] != 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) open += __shfl_xor_sync(0xffffffffu, open, o);
        if ((tid & 31) == 0) atomicAdd(&s_open, open);
    }

    // ---- 2. mark the solution (goal -> start along BFS parents); D = decision cells on it
    if (tid == 0) {
        int b = goal_idx, dcount = 0, junctions = 0, crossings = 0, turns = 0, arrived = 0;
        for (;;) {
            const int ci = block_cell(b);
            ms.flags[ci] |= MF_SOL;
            const int nbc = ms.flags[ci] & MF_NB;
            if (nbc > 2) ++dcount;   // metrics_calculator.py:71-85 (only cells can have > 2)
            junctions += nbc == 3;   // calculate_J :39-53
            crossings += nbc == 4;   // calculate_CR :55-69
            if (b == start_idx) break;
            const int step = offs[ms.flags[ci] >> MF_PDIR_SHIFT];
            if (arrived != 0 && arrived != step) ++turns;   // calculate_T :28-37 (interior blocks only; passages are straight)
            arrived = step;
            b += 2 * step;   // passage block, then the next cell
        }
        s_dcount = dcount;
        s_sol_counts[0] = turns; s_sol_counts[1] = junctions; s_sol_counts[2] = crossings;
    }
    __syncthreads();

    // ---- 3. parent node and edge length of every node (walk straight up to the next node)
    for (int ci = tid; ci < cells; ci += nthr) {
        if (!(ms.flags[ci] & MF_NODE) || ci == start_c) continue;
        int b = cell_block(ci);
        const int step = offs[ms.flags[ci] >> MF_PDIR_SHIFT];
        int hops = 0, pc;
        do {
            b += 2 * step;
            ++hops;
            pc = block_cell(b);
        } while (!(ms.flags[pc] & MF_NODE));
        ms.pnode[ci] = (unsigned short)pc;
        // low byte: blocks strictly between (maze_complexity_evaluation.py:176-184); bits 8-9: direction towards the parent
        const int dcode = step == -Wb ? 0 : (step == Wb ? 1 : (step == -1 ? 2 : 3));
        ms.dpar[ci] = (unsigned short)((2 * hops - 1) | (dcode << 8));
    }
    __syncthreads();

    auto is_sol = [&](int ci) { return (ms.flags[ci] & MF_SOL) != 0; };
    auto nbof = [&](int ci) { return ms.flags[ci] & MF_NB; };
    auto is_plain = [&](int ci) { return !is_sol(ci) && nbof(ci) != 3; };
    auto is_dead_end_off = [&](int ci) { return (ms.flags[ci] & MF_NODE) && nbof(ci) == 1 && !is_sol(ci); };

    // ---- 4. Kim-Crawfis DE (metrics_calculator.py:87-173).  Whether a dead end counts depends on the
    // decision points recorded by the dead ends before it in row-major order, so the final pass is
    // sequential; everything that does not depend on that order is done in parallel first:
    //   4a  nearest node with more than two open neighbours above every node (ms.minleaf as scratch)
    //   4b  per dead end: cut or not, alcove / forward / backward (ms.comp as scratch)
    //   4c  thread 0: walk only the chain of decision points above each dead end, stop at the first
    //       recorded one
    int alcoves = 0, forward = 0, backward = 0;
    double x_lde = 0.0, x_t[3] = {0.0, 0.0, 0.0}, x_d[3] = {0.0, 0.0, 0.0}, x_l[3] = {0.0, 0.0, 0.0};
    const double ce_d = (double)((Hb - 1) * ((Wb - 1) / 2) - 1);   // metrics_calculator.py:16
    if (with_kc) {
        unsigned short* jup = ms.minleaf;
        unsigned short* kind = ms.comp;
        auto dcode = [&](int ci) { return (ms.dpar[ci] >> 8) & 3; };
        for (int ci = tid; ci < cells; ci += nthr) {
            if (!(ms.flags[ci] & MF_NODE)) continue;
            int y = ms.pnode[ci];
            while (y != 0xffff && (ms.flags[y] & MF_NB) <= 2) y = ms.pnode[y];
            jup[ci] = (unsigned short)y;
        }
        __syncthreads();
        const int gr = goal_idx / Wb, gc = goal_idx % Wb;
        for (int de = tid; de < cells; de += nthr) {
            if (!is_dead_end_off(de)) continue;
            // attachment A = first solution node above; cut iff it sits at path index <= sol_len - 2
            int a = ms.pnode[de];
            while (!is_sol(a)) a = ms.pnode[a];
            const int db = cell_block(de);
            const int j = (int)f.dist[db] - (int)f.dist[cell_block(a)];
            const bool cut = j <= sol_len - 2;
            // interior nodes: strictly above the dead end, up to (cut) the node below A or (uncut) the node below start
            bool has_turn = false;
            int prev = de, below_a = de, n_turns = 0, n_dp = 0;
            for (int y = ms.pnode[de]; cut ? (y != a) : (y != start_c); y = ms.pnode[y]) {
                if (dcode(prev) != dcode(y)) { has_turn = true; ++n_turns; }
                n_dp += (ms.flags[y] & MF_NB) > 2;
                if (!is_sol(y)) below_a = y;
                prev = y;
            }
            const int fj = jup[de];
            const bool has_dp = fj != 0xffff && (cut ? !is_sol(fj) : fj != start_c);
            const int len = cut ? j : (int)f.dist[db] + 1;
            int k = 0;   // 0 alcove, 1 forward, 2 backward (type_of_DE :153-173)
            if (len >= 3 && (has_turn || has_dp)) {
                int lr, lc;   // path[-1]
                if (cut) {
                    const int back[4] = {Wb, -Wb, 1, -1};   // from A one block towards the node below it
                    const int ab = cell_block(a) + back[dcode(below_a)];
                    lr = ab / Wb; lc = ab % Wb;
                } else {
                    lr = start_idx / Wb; lc = start_idx % Wb;
                }
                const int diff = (abs(lr - gr) + abs(lc - gc)) - (abs(db / Wb - gr) + abs(db % Wb - gc));
                k = diff > 0 ? 1 : 2;
            }
            kind[de] = (unsigned short)(k | (cut ? 4 : 0));
            if (ext) {   // per dead end terms of T_DE :175-185, D_sharp :187-197, L_sharp / L_DE :199-241
                if (!cut && (ms.flags[start_c] & MF_NB) > 2) ++n_dp;   // an uncut path ends on start itself
                ms.dsum[de] = (unsigned)len;
                ms.ssum[de] = __ddiv_rn(__ddiv_rn((double)n_turns, (double)sol_len), (double)len);
                ms.bsum[de] = __ddiv_rn(__ddiv_rn((double)n_dp, (double)sol_len), (double)len);
            }
        }
        __syncthreads();
        // 4c.  The reference walks the dead ends in row-major order: dead end d counts unless a decision point of
        // its chain was recorded by an earlier counted dead end, and a counted dead end records the first decision
        // point of its chain.  With rec[P] = smallest index of a counted dead end whose first decision point is P,
        //     counted(d)  <=>  no P in chain(d) has rec[P] < d,
        // and this system has exactly one solution (by induction on d, which only looks at smaller indices).  It is
        // reached by iterating from "everything counts": after k rounds the k smallest dead ends are final, in
        // practice a handful of rounds; a round without a change is the fixpoint.  (The sequential pass this
        // replaces was 66 % of the kernel's time on r-prim mazes.)  rec lives in ms.dsum at decision-point cells;
        // the ext sums keep their terms in ms.dsum / ssum / bsum at dead-end cells, which are different cells.
        constexpr unsigned NOT_RECORDED = 0xffffffffu;
        constexpr int COUNTED = 8;
        auto in_range = [&](int y, bool cut) { return y != 0xffff && (cut ? !is_sol(y) : y != start_c); };
        for (int ci = tid; ci < cells; ci += nthr)
            if (is_dead_end_off(ci)) kind[ci] |= COUNTED;
        // (bounded on purpose: at most one round per dead end is ever needed, and an unbounded `for (;;)` around
        // the barrier-with-reduction died with "illegal instruction" on 41 x 41 mazes on sm_100a, CUDA 12.9)
        for (int round = 0; round <= cells; ++round) {
            for (int ci = tid; ci < cells; ci += nthr)
                if ((ms.flags[ci] & MF_NODE) && nbof(ci) > 2) ms.dsum[ci] = NOT_RECORDED;
            __syncthreads();
            for (int de = tid; de < cells; de += nthr) {
                if (!is_dead_end_off(de) || !(kind[de] & COUNTED)) continue;
                const int f = jup[de];
                if (in_range(f, (kind[de] & 4) != 0)) atomicMin(&ms.dsum[f], (unsigned)de);
            }
            __syncthreads();
            int changed = 0;
            for (int de = tid; de < cells; de += nthr) {
                if (!is_dead_end_off(de)) continue;
                const int kd = kind[de];
                const bool cut = (kd & 4) != 0;
                bool blocked = false;
                for (int y = jup[de]; in_range(y, cut); y = jup[y])
                    if (ms.dsum[y] < (unsigned)de) { blocked = true; break; }
                if (blocked == ((kd & COUNTED) != 0)) {
                    kind[de] = (unsigned short)(kd ^ COUNTED);
                    changed = 1;
                }
            }
            if (!__syncthreads_or(changed)) break;
        }
        {
            int na = 0, nf = 0, nb_ = 0;
            for (int de = tid; de < cells; de += nthr) {
                if (!is_dead_end_off(de) || !(kind[de] & COUNTED)) continue;
                const int k = kind[de] & 3;
                na += k == 0; nf += k == 1; nb_ += k == 2;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                na += __shfl_xor_sync(0xffffffffu, na, o);
                nf += __shfl_xor_sync(0xffffffffu, nf, o);
                nb_ += __shfl_xor_sync(0xffffffffu, nb_, o);
            }
            if ((tid & 31) == 0) { atomicAdd(&s_de_counts[0], na); atomicAdd(&s_de_counts[1], nf); atomicAdd(&s_de_counts[2], nb_); }
        }
        if (ext && tid == 0) {   // sums over ALL off-solution dead ends, in row-major order (float sums: order matters)
            for (int de = 0; de < cells; ++de) {
                if (!is_dead_end_off(de)) continue;
                const int k = kind[de] & 3;
                const double l = __ddiv_rn((double)ms.dsum[de], ce_d);
                x_lde = __dadd_rn(x_lde, l);
                x_l[k] = __dadd_rn(x_l[k], l);
                x_t[k] = __dadd_rn(x_t[k], ms.ssum[de]);
                x_d[k] = __dadd_rn(x_d[k], ms.bsum[de]);
            }
        }
        __syncthreads();
        alcoves = s_de_counts[0]; forward = s_de_counts[1]; backward = s_de_counts[2];
        for (int ci = tid; ci < cells; ci += nthr) {   // scratch back to its initial state
            ms.minleaf[ci] = 0xffffu; ms.comp[ci] = 0xffffu;
            ms.dsum[ci] = 0u;   // held rec[] at decision points (and the ext terms at dead ends)
            if (ext) { ms.ssum[ci] = 0.0; ms.bsum[ci] = 0.0; }
        }
        __syncthreads();
    }

    // ---- 5. smallest dead-end rank below every off-solution node (adjacency order of the reference)
    for (int ci = tid; ci < cells; ci += nthr) {
        if (!is_dead_end_off(ci)) continue;
        // A walk stops at the first node that already holds a smaller rank: the dead end that put it there is
        // on its own way up and covers every ancestor (the smallest rank of a subtree never meets a smaller one
        // inside it, so it always reaches the subtree's root).  Without the early exit every walk hammered the
        // same few nodes next to the solution with CAS loops (22 % of the kernel on r-prim mazes).
        int y = ci;
        while (!is_sol(y)) {
            if (!atomic_min_u16(ms.minleaf + y, (unsigned short)ci)) break;
            y = ms.pnode[y];
        }
    }
    // ---- 6. component root of every plain node
    for (int ci = tid; ci < cells; ci += nthr) {
        if (!(ms.flags[ci] & MF_NODE) || !is_plain(ci)) continue;
        int r = ci;
        while (is_plain(ms.pnode[r])) r = ms.pnode[r];
        ms.comp[ci] = (unsigned short)r;
    }
    __syncthreads();

    // ---- 7. every tree edge goes to at most one hallway (maze_complexity_evaluation.py:186-221)
    for (int n = tid; n < cells; n += nthr) {
        if (!(ms.flags[n] & MF_NODE) || n == start_c) continue;
        const int p = ms.pnode[n];
        const unsigned d = ms.dpar[n] & 0xffu;
        const double s = 1.0 / (double)(2 * d);
        if (is_sol(n)) {                       // solution chain = hallway 0
            atomicAdd(&s_D0, (double)d);
            atomicAdd(&s_S0, s);
        } else if (nbof(n) != 3) {             // plain child
            if (is_plain(p) || nbof(p) == 3) {
                atomicAdd(&ms.dsum[ms.comp[n]], d);
                atomicAdd(&ms.ssum[ms.comp[n]], s);
            }
        } else if (is_plain(p)) {              // off-solution junction below a plain node
            const int pp = ms.pnode[p];
            const bool broke = nbof(pp) == 3 && is_sol(pp);   // :209-214 `break`
            if (!broke || ms.minleaf[n] == ms.minleaf[p]) {
                atomicAdd(&ms.dsum[ms.comp[p]], d);
                atomicAdd(&ms.ssum[ms.comp[p]], s);
            }
        }
    }
    __syncthreads();

    // ---- 8. hallway complexity -> branch (maze_complexity_evaluation.py:223-259,286-308)
    for (int r = tid; r < cells; r += nthr) {
        if (!(ms.flags[r] & MF_NODE) || ms.comp[r] != r) continue;
        const double c = (double)ms.dsum[r] * ms.ssum[r];
        int below = r, x = ms.pnode[r];
        while (!is_sol(x)) { below = x; x = ms.pnode[x]; }
        int key = below;
        if (nbof(x) == 3) {                    // junction on the solution: key = head of its junction run
            key = x;
            while (key != start_c && nbof(ms.pnode[key]) == 3) key = ms.pnode[key];
        }
        atomicAdd(&ms.bsum[key], c);
    }
    __syncthreads();

    // ---- 9. reduce: sum and product over branches
    double tsum = 0.0, tprod = 1.0;
    for (int k = tid; k < cells; k += nthr) {
        const double v = ms.bsum[k];
        tsum += v;
        tprod *= v + 1.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
        tprod *= __shfl_xor_sync(0xffffffffu, tprod, o);
    }
    if ((tid & 31) == 0) { s_red[0][tid >> 5] = tsum; s_red[1][tid >> 5] = tprod; }
    __syncthreads();
    if (tid == 0) {
        double sum = 0.0, prod = 1.0;
        for (int w = 0; w < nthr / 32; ++w) { sum += s_red[0][w]; prod *= s_red[1][w]; }
        const double c0 = s_D0 * s_S0;
        out.difficulty = log(c0 * prod);       // :319-329
        out.complexity = log(c0 + sum);        // :310-317
        const double ce = (double)((Hb - 1) * ((Wb - 1) / 2) - 1);   // metrics_calculator.py:16
        out.L = __ddiv_rn((double)sol_len, ce);
        out.D = __ddiv_rn((double)s_dcount, (double)sol_len);
        out.DE = __dadd_rn(__dadd_rn(__ddiv_rn((double)alcoves, (double)sol_len), __ddiv_rn((double)forward, (double)sol_len)),
                           __ddiv_rn((double)backward, (double)sol_len));   // AC + FDE + BDE, :97-98
        out.sol_len = sol_len;
        out.de_count = alcoves + forward + backward;
        if (ext) {
            const double sl = (double)sol_len;
            out.ext[MAZE_METRIC_EXT_DENSITY] = __ddiv_rn((double)s_open, (double)(Hb * Wb));
            out.ext[MAZE_METRIC_EXT_T] = __ddiv_rn((double)s_sol_counts[0], sl);
            out.ext[MAZE_METRIC_EXT_J] = __ddiv_rn((double)s_sol_counts[1], sl);
            out.ext[MAZE_METRIC_EXT_CR] = __ddiv_rn((double)s_sol_counts[2], sl);
            out.ext[MAZE_METRIC_EXT_AC] = __ddiv_rn((double)alcoves, sl);
            out.ext[MAZE_METRIC_EXT_FDE] = __ddiv_rn((double)forward, sl);
            out.ext[MAZE_METRIC_EXT_BDE] = __ddiv_rn((double)backward, sl);
            out.ext[MAZE_METRIC_EXT_L_DE] = x_lde;
            for (int k = 0; k < 3; ++k) {
                out.ext[MAZE_METRIC_EXT_T_DE + k] = x_t[k];
                out.ext[MAZE_METRIC_EXT_D_SHARP + k] = x_d[k];
                out.ext[MAZE_METRIC_EXT_L_SHARP + k] = x_l[k];
            }
            for (int k = MAZE_METRIC_EXT_L_SHARP + 3; k < MAZE_METRIC_EXT_WORDS; ++k) out.ext[k] = 0.0;
        }
    }
    __syncthreads();
}
