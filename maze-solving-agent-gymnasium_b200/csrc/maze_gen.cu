// Batched maze generation on the device (sm_100a): r-prim, dfs, prim&kill + goal selection +
// per-maze fields (step table, step budget).
//
// A maze of N x N logical cells (N <= 64) is held as two wall bit-planes in the REGISTERS of one
// warp: E (bit j of row i = open passage between cells (i, j) and (i, j+1)) and S (between (i, j)
// and (i+1, j)), one 64-bit word per lattice row, rows l and l+32 in lane l.  Cell sets (in-tree,
// frontier, visited, marked) use the same layout, so "pick a uniformly random frontier cell" is
// popcount + warp scan + ballot, and a breadth-first level over the whole lattice is a handful of
// shifts and four shuffles regardless of the frontier size.
//
//   maze_generate_warp_kernel   one WARP per maze, no shared memory: generation, goal selection
//                               (BFS from start), BFS from the goal recording parent direction /
//                               level parity / far flag as bit-planes, then the block grid and the
//                               one-byte-per-block step table are written straight from registers.
//                               Bordered (euclidean) mazes without difficulty scoring: the
//                               throughput path (many warps per SM hide the dependent-issue latency
//                               of the sequential carving loop).
//   maze_generate_kernel        one CTA per maze, block grid staged in shared memory: toroidal
//                               mazes (the seam links passage blocks to passage blocks, so fields
//                               need a block-resolution BFS) and scored generation (best-of-k by
//                               McClendon difficulty).  Same generators, hence the same mazes.
//
// Reference: lib/maze_generation.py:6-35 (gen_maze), :37-56 (gen_maze_no_border), :59-99 (r-prim),
// :101-128 (dfs), :130-185 (prim&kill), :187-218 (goal = farthest leaf, row-major tie-break).
// RNG: PCG32 seeded by Philox4x32-10 keyed by (seed, global slot id, generation count, candidate) -- the reference
// draws from Python's global `random` through set iteration order, which cannot be replayed, so
// parity with the reference is distributional: exact output distributions on small lattices
// (oracle/gen_exact.py), and every maze bit-exact against a model of this stream (oracle/gen_stream.py).
#include "maze_metrics.cuh"
#include "maze_walls.cuh"

namespace {

constexpr int GEN_THREADS = METRIC_THREADS;   // CTA-per-maze kernel (scores with maze_metrics)
constexpr int WARP_GEN_THREADS = 256;        // warp-per-maze kernel: 8 mazes per CTA

struct GenParams {
    uint8_t* grids;          // [M, slot] out (may be NULL)
    int32_t* meta;           // [M, 8] in: H, W, FLAGS ; out: START, GOAL, MAX_STEPS, SOL_LEN, SPARE(gen count)
    uint8_t* table;          // [M, slot] out
    const int32_t* ids;      // [n] slots to generate (NULL = 0..n-1)
    const int32_t* count_dev;// optional device-side n
    int n;
    int slot;
    int smem_hw;
    int smem_cells;          // 0 when no metrics are needed
    int candidates;          // best-of-k by McClendon difficulty (base_maze_env.py:78-97); 1 = raw generator
    int candidate_base;      // test hook (MAZE_GEN_CANDIDATE_BASE): RNG key of candidate c is candidate_base + c
    int only_toroidal;       // CTA kernel: skip bordered slots (the warp kernel did them)
    int* work_counter;       // warp kernel: next unclaimed item (mazes differ in cost: claim dynamically)
    double* difficulty;      // [n] optional out: difficulty of the maze kept for item k
    unsigned long long seed;
    long long slot_id_base;
    // scored bulk generation in two kernels: candidate wall planes drawn by the warp kernel into scratch
    unsigned long long* planes;   // [n * candidates, PLANE_WORDS] or NULL
    int item_base;                // first item of this chunk when ids is NULL
};

// one candidate in scratch: E plane (64 rows), S plane (64 rows), then start / goal cell
constexpr int PLANE_WORDS = 2 * MAZE_GEN_MAX_CELLS + 2;

// Per-maze random stream: PCG-XSH-RR 64/32 whose state and increment come from one Philox4x32-10
// block keyed by (seed, global slot id | generation count, candidate).  The key makes streams
// independent of how slots are sharded over GPUs; the sequential generator costs ~12 instructions
// per draw inside the carving loop (a Philox block per two draws was 20 % of the kernel).
struct GenRng {
    u64 state, inc;
    __device__ __forceinline__ void init(unsigned long long seed, u64 seq, unsigned sub) {
        Philox p;
        p.init(seed, seq, sub);
        p.refill();
        state = ((u64)p.o1 << 32) | p.o0;
        inc = ((((u64)p.o3 << 32) | p.o2) << 1) | 1ull;
        next();
    }
    __device__ __forceinline__ unsigned next() {
        const u64 old = state;
        state = old * 6364136223846793005ull + inc;
        const unsigned xs = (unsigned)(((old >> 18) ^ old) >> 27);
        return __funnelshift_r(xs, xs, (unsigned)(old >> 59));
    }
    __device__ __forceinline__ unsigned below(unsigned n) { return __umulhi(next(), n); }   // bias < n / 2^32
};

__device__ __forceinline__ int warp_incl_scan(int v) {
    const int lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(FULL, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// k-th (0-based) set bit of a warp-uniform 64-bit word, found by all lanes at once
__device__ __forceinline__ int select64_warp(u64 w, int k) {
    const int lane = lane_id();
    const unsigned lo = (unsigned)w, hi = (unsigned)(w >> 32);
    const int plo = __popc(lo);
    const bool upper = k >= plo;
    const unsigned m = upper ? hi : lo;
    const int kk = upper ? k - plo : k;
    const bool hit = ((m >> lane) & 1u) && __popc(m & ((1u << lane) - 1u)) == kk;
    return (upper ? 32 : 0) + __ffs(__ballot_sync(FULL, hit)) - 1;
}

// uniformly random set bit over the two rows of all lanes; returns (i << 8) | j, or -1 if empty
__device__ __forceinline__ int pick_uniform(u64 s0, u64 s1, GenRng& rng) {
    const int c0 = __popcll(s0), c1 = __popcll(s1);
    const int incl = warp_incl_scan(c0 + c1);
    const int total = __shfl_sync(FULL, incl, 31);
    if (total == 0) return -1;
    const int k = (int)rng.below((unsigned)total);
    const int owner = __ffs(__ballot_sync(FULL, incl > k)) - 1;
    int kk = k - __shfl_sync(FULL, incl - c0 - c1, owner);
    const u64 w0 = __shfl_sync(FULL, s0, owner), w1 = __shfl_sync(FULL, s1, owner);
    const int n0 = __popcll(w0);
    const bool second = kk >= n0;
    if (second) kk -= n0;
    return ((owner + (second ? 32 : 0)) << 8) | select64_warp(second ? w1 : w0, kk);
}

// 4-bit mask of lattice neighbours of (i, j) whose bit in `s` equals `want`:
// bit0 up (i-1), bit1 down (i+1), bit2 left (j-1), bit3 right (j+1); out-of-lattice never counts
__device__ __forceinline__ unsigned neighbour_mask(const RowSets& s, int i, int j, int nr, int nc, bool want) {
    const u64 w = want ? 1ull : 0ull;
    unsigned nb = 0;
    if (i > 0 && ((row_get(s, i - 1) >> j) & 1ull) == w) nb |= 1u;
    if (i + 1 < nr && ((row_get(s, i + 1) >> j) & 1ull) == w) nb |= 2u;
    const u64 r = row_get(s, i);
    if (j > 0 && ((r >> (j - 1)) & 1ull) == w) nb |= 4u;
    if (j + 1 < nc && ((r >> (j + 1)) & 1ull) == w) nb |= 8u;
    return nb;
}

// index of the k-th set bit of a 4-bit mask (64-entry, 2-bit look-up table in two constants)
__device__ __forceinline__ int select4(unsigned nb, int k) {
    const int idx = (int)nb * 4 + k;
    const u64 t = idx < 32 ? 0x2409080204010000ull : 0xe439380e340d0c03ull;
    return (int)((t >> (2 * (idx & 31))) & 3ull);
}
__device__ __forceinline__ int pick_direction(unsigned nb, GenRng& rng) {
    return select4(nb, (int)rng.below((unsigned)__popc(nb)));
}

__device__ __forceinline__ void dir_delta(int d, int& di, int& dj) {   // 0 up 1 down 2 left 3 right
    di = (d == 1) - (d == 0);
    dj = (d == 3) - (d == 2);
}

// open the wall of cell (i, j) towards direction d
__device__ __forceinline__ void open_wall(Walls& w, int i, int j, int d) {
    if (d < 2) row_or(w.s, d == 0 ? i - 1 : i, 1ull << j);
    else row_or(w.e, i, 1ull << (d == 2 ? j - 1 : j));
}

// ---- generators (all 32 lanes, uniform control flow) -----------------------------------------

// lib/maze_generation.py:59-99: uniformly random frontier cell, then a uniformly random tree neighbour
__device__ __forceinline__ void gen_random_prim(Walls& w, int nr, int nc, int si, int sj, GenRng& rng) {
    const int lane = lane_id();
    const u64 colmask = nc >= 64 ? ~0ull : ((1ull << nc) - 1ull);
    RowSets in = {0ull, 0ull}, fr = {0ull, 0ull};
    auto add_cell = [&](int i, int j) {
        const u64 bit = 1ull << j;
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
            const int row = lane + 32 * sl;
            u64& w_in = sl ? in.a1 : in.a0;
            u64& w_fr = sl ? fr.a1 : fr.a0;
            if (row >= nr) continue;
            if (row == i) {
                w_in |= bit;
                w_fr &= ~bit;
                w_fr |= ((bit << 1) | (bit >> 1)) & ~w_in & colmask;
            } else if (row == i - 1 || row == i + 1) {
                w_fr |= bit & ~w_in;
            }
        }
    };
    add_cell(si, sj);
    for (;;) {
        const int p = pick_uniform(fr.a0, fr.a1, rng);
        if (p < 0) break;
        const int i = p >> 8, j = p & 0xff;
        const unsigned nb = neighbour_mask(in, i, j, nr, nc, true);   // never empty for a frontier cell
        open_wall(w, i, j, pick_direction(nb, rng));
        add_cell(i, j);
    }
}

// lib/maze_generation.py:101-128 (first unvisited neighbour of a fresh shuffle == uniform choice).
// The explicit stack is replaced by a 2-bit "direction back to the parent" plane: popping the
// stack is walking to the parent.
__device__ __forceinline__ void gen_depth_first(Walls& w, int nr, int nc, int si, int sj, GenRng& rng) {
    RowSets vis = {0ull, 0ull}, b0 = {0ull, 0ull}, b1 = {0ull, 0ull};
    row_or(vis, si, 1ull << sj);
    int i = si, j = sj;
    for (;;) {
        const unsigned nb = neighbour_mask(vis, i, j, nr, nc, false);
        int di, dj;
        if (nb) {
            const int d = pick_direction(nb, rng);
            dir_delta(d, di, dj);
            i += di; j += dj;
            const int back = d ^ 1;
            open_wall(w, i, j, back);
            row_or(vis, i, 1ull << j);
            if (back & 1) row_or(b0, i, 1ull << j);
            if (back & 2) row_or(b1, i, 1ull << j);
        } else {
            if (i == si && j == sj) break;
            dir_delta(cell_bit(b0, i, j) | (cell_bit(b1, i, j) << 1), di, dj);
            i += di; j += dj;
        }
    }
}

// lib/maze_generation.py:130-185
__device__ __forceinline__ void gen_prim_and_kill(Walls& w, int nr, int nc, int si, int sj, GenRng& rng) {
    const int lane = lane_id();
    const u64 colmask = nc >= 64 ? ~0ull : ((1ull << nc) - 1ull);
    // marked rows; bits / rows outside the lattice read as "marked" so they never look eligible
    RowSets mk;
    mk.a0 = lane < nr ? ~colmask : ~0ull;
    mk.a1 = lane + 32 < nr ? ~colmask : ~0ull;
    row_or(mk, si, 1ull << sj);
    int unmarked = nr * nc - 1;
    int i = si, j = sj;
    for (;;) {
        // random walk until no unmarked neighbour (:154-185)
        for (;;) {
            const unsigned nb = neighbour_mask(mk, i, j, nr, nc, false);
            if (!nb) break;
            const int d = pick_direction(nb, rng);
            int di, dj;
            dir_delta(d, di, dj);
            i += di; j += dj;
            open_wall(w, i, j, d ^ 1);
            row_or(mk, i, 1ull << j);
            --unmarked;
        }
        if (unmarked == 0) break;
        // restart from a uniformly random marked cell with an unmarked neighbour (:150-152)
        u64 up0 = __shfl_up_sync(FULL, mk.a0, 1);
        u64 up1 = __shfl_up_sync(FULL, mk.a1, 1);
        const u64 last0 = __shfl_sync(FULL, mk.a0, 31);
        if (lane == 0) { up0 = ~0ull; up1 = last0; }
        u64 dn0 = __shfl_down_sync(FULL, mk.a0, 1);
        u64 dn1 = __shfl_down_sync(FULL, mk.a1, 1);
        const u64 first1 = __shfl_sync(FULL, mk.a1, 0);
        if (lane == 31) { dn0 = first1; dn1 = ~0ull; }
        const u64 e0 = mk.a0 & colmask & (~up0 | ~dn0 | (~mk.a0 << 1) | (~mk.a0 >> 1));
        const u64 e1 = mk.a1 & colmask & (~up1 | ~dn1 | (~mk.a1 << 1) | (~mk.a1 >> 1));
        const int p = pick_uniform(lane < nr ? e0 : 0ull, lane + 32 < nr ? e1 : 0ull, rng);
        if (p < 0) break;   // cannot happen on a connected lattice
        i = p >> 8; j = p & 0xff;
    }
}

// gen_maze's random part (lib/maze_generation.py:21-30): start cell + generator.  Identical in
// both kernels, so a slot's candidate c is the same maze whichever kernel draws it.
__device__ __forceinline__ void generate_walls(Walls& w, int algo, int nr, int nc, unsigned long long seed, u64 seq,
                                               unsigned cand, int& si, int& sj) {
    GenRng rng;
    rng.init(seed, seq, cand);
    si = (int)rng.below((unsigned)nr);   // :21 uniform logical cell
    sj = (int)rng.below((unsigned)nc);
    w.e.a0 = w.e.a1 = w.s.a0 = w.s.a1 = 0ull;
    if (algo == MAZE_ALGO_RPRIM) gen_random_prim(w, nr, nc, si, sj, rng);
    else if (algo == MAZE_ALGO_DFS) gen_depth_first(w, nr, nc, si, sj, rng);
    else gen_prim_and_kill(w, nr, nc, si, sj, rng);
}

// goal = the leaf farthest from start, first in row-major order on ties
// (lib/maze_generation.py:187-218); returns (gi << 8) | gj
__device__ __forceinline__ int select_goal(const Walls& w, int si, int sj) {
    const int lane = lane_id();
    // leaves: exactly one open wall
    const u64 su0 = __shfl_up_sync(FULL, w.s.a0, 1), su1 = __shfl_up_sync(FULL, w.s.a1, 1), swrap = __shfl_sync(FULL, w.s.a0, 31);
    u64 leaf0, leaf1;
    {
        const u64 L = w.e.a0 << 1, R = w.e.a0, U = lane == 0 ? 0ull : su0, D = w.s.a0;
        leaf0 = (L ^ R ^ U ^ D) & ~((L & R) | (L & U) | (L & D) | (R & U) | (R & D) | (U & D));
    }
    {
        const u64 L = w.e.a1 << 1, R = w.e.a1, U = lane == 0 ? swrap : su1, D = w.s.a1;
        leaf1 = (L ^ R ^ U ^ D) & ~((L & R) | (L & U) | (L & D) | (R & U) | (R & D) | (U & D));
    }
    u64 f0 = 0ull, f1 = 0ull;
    if ((si & 31) == lane) { if (si >> 5) f1 = 1ull << sj; else f0 = 1ull << sj; }
    u64 v0 = f0, v1 = f1, best0 = 0ull, best1 = 0ull;
    for (;;) {
        Reach x;
        bfs_expand(w, f0, f1, x);
        const u64 n0 = (x.l0 | x.r0 | x.a0 | x.b0) & ~v0, n1 = (x.l1 | x.r1 | x.a1 | x.b1) & ~v1;
        if (!__ballot_sync(FULL, (n0 | n1) != 0ull)) break;
        v0 |= n0; v1 |= n1; f0 = n0; f1 = n1;
        const u64 lf0 = n0 & leaf0, lf1 = n1 & leaf1;
        if (__ballot_sync(FULL, (lf0 | lf1) != 0ull)) { best0 = lf0; best1 = lf1; }
    }
    const unsigned has0 = __ballot_sync(FULL, best0 != 0ull), has1 = __ballot_sync(FULL, best1 != 0ull);
    if (!(has0 | has1)) return (si << 8) | sj;   // one-cell lattice
    const int owner = has0 ? __ffs(has0) - 1 : __ffs(has1) - 1;
    const u64 word = __shfl_sync(FULL, has0 ? best0 : best1, owner);
    return ((owner + (has0 ? 0 : 32)) << 8) | (__ffsll((long long)word) - 1);
}

struct GoalField {   // what the step table needs, as bit-planes over the cell lattice
    RowSets p0, p1;   // action code (2 bits) of the move from a cell towards its parent (towards the goal)
    RowSets q;        // parity of the cell's level (distance to the goal in cells)
    RowSets f;        // "far": block distance 2 * level > L (the depth-limited A* of the reference gives up)
    int start_level;
};

__device__ __forceinline__ void goal_field(const Walls& w, int gi, int gj, int si, int sj, int L, GoalField& g) {
    const int lane = lane_id();
    g.p0 = g.p1 = g.q = g.f = RowSets{0ull, 0ull};
    g.start_level = 0;
    u64 f0 = 0ull, f1 = 0ull;
    if ((gi & 31) == lane) { if (gi >> 5) f1 = 1ull << gj; else f0 = 1ull << gj; }
    u64 v0 = f0, v1 = f1;
    const u64 sbit0 = ((si & 31) == lane && !(si >> 5)) ? 1ull << sj : 0ull;
    const u64 sbit1 = ((si & 31) == lane && (si >> 5)) ? 1ull << sj : 0ull;
    for (int level = 1;; ++level) {
        Reach x;
        bfs_expand(w, f0, f1, x);
        const u64 n0 = (x.l0 | x.r0 | x.a0 | x.b0) & ~v0, n1 = (x.l1 | x.r1 | x.a1 | x.b1) & ~v1;
        if (!__ballot_sync(FULL, (n0 | n1) != 0ull)) break;
        // parent above -> move up (1), below -> down (0), right -> right (2), left -> left (3)
        g.p0.a0 |= n0 & (x.a0 | x.l0);  g.p0.a1 |= n1 & (x.a1 | x.l1);
        g.p1.a0 |= n0 & (x.r0 | x.l0);  g.p1.a1 |= n1 & (x.r1 | x.l1);
        if (level & 1) { g.q.a0 |= n0; g.q.a1 |= n1; }
        if (2 * level > L) { g.f.a0 |= n0; g.f.a1 |= n1; }
        if (__ballot_sync(FULL, ((n0 & sbit0) | (n1 & sbit1)) != 0ull)) g.start_level = level;
        v0 |= n0; v1 |= n1; f0 = n0; f1 = n1;
    }
}

// Block grid + step table of a bordered maze, written row by row from the register planes.
// Closed form of base_maze_env.py:224-262 on a tree (oracle/grid.py:best_dir_code_table): the
// neighbour on the way to the goal wins while the block is within the A* depth limit; beyond it
// (and on the goal itself) all neighbours tie on path length and plain Manhattan distance decides,
// first in action order (down, up, right, left).
__device__ __forceinline__ void encode_bordered(const Walls& w, const GoalField& g, int H, int W, int gi, int gj,
                                                uint8_t* __restrict__ table, uint8_t* __restrict__ grid) {
    const int lane = lane_id();
    const int gr = 2 * gi + 1, gc = 2 * gj + 1;
    for (int r = 0; r < H; ++r) {
        const bool cell_row = (r & 1) != 0;
        const int i = cell_row ? (r - 1) >> 1 : (r >> 1) - 1;   // cell row, or the cell row above a passage row
        const bool inner = r > 0 && r < H - 1;
        u64 Ei = 0, Si = 0, Su = 0, P0i = 0, P1i = 0, Qi = 0, Fi = 0, P0n = 0, P1n = 0, Qn = 0, Fn = 0;
        if (inner) {
            Si = row_get(w.s, i); P0i = row_get(g.p0, i); P1i = row_get(g.p1, i); Qi = row_get(g.q, i); Fi = row_get(g.f, i);
            if (cell_row) {
                Ei = row_get(w.e, i);
                if (i > 0) Su = row_get(w.s, i - 1);
            } else {
                P0n = row_get(g.p0, i + 1); P1n = row_get(g.p1, i + 1); Qn = row_get(g.q, i + 1); Fn = row_get(g.f, i + 1);
            }
        }
        for (int c = lane; c < W; c += 32) {
            int tab = 0, gv = 0;
            if (inner && c > 0 && c < W - 1) {
                if (cell_row && (c & 1)) {                       // logical cell (i, j)
                    const int j = (c - 1) >> 1;
                    const bool is_goal = (i == gi) && (j == gj);
                    int code;
                    if (!is_goal && !((Fi >> j) & 1ull)) {
                        code = (int)((P0i >> j) & 1ull) | ((int)((P1i >> j) & 1ull) << 1);
                    } else {
                        const int open_a[4] = {(int)((Si >> j) & 1ull), (int)((Su >> j) & 1ull), (int)((Ei >> j) & 1ull),
                                               j > 0 ? (int)((Ei >> (j - 1)) & 1ull) : 0};
                        int best = 0x7fffffff;
                        code = 4;
#pragma unroll
                        for (int a = 0; a < 4; ++a) {
                            int dr, dc;
                            action_delta(a, dr, dc);
                            const int man = abs(r + dr - gr) + abs(c + dc - gc);
                            if (open_a[a] && man < best) { best = man; code = a; }
                        }
                    }
                    tab = MAZE_TAB_OPEN | (code << MAZE_TAB_CODE_SHIFT) | ((int)((Qi >> j) & 1ull) << (MAZE_TAB_D4_SHIFT + 1));
                    gv = is_goal ? 2 : 1;
                } else if (cell_row) {                           // passage between (i, j) and (i, j + 1)
                    const int j = (c - 2) >> 1;
                    if ((Ei >> j) & 1ull) {
                        const bool child_right = ((P0i >> (j + 1)) & 1ull) && ((P1i >> (j + 1)) & 1ull);   // its parent is on the left
                        const int jc = child_right ? j + 1 : j;
                        const int code = ((Fi >> jc) & 1ull) ? (c < gc ? 2 : 3) : (child_right ? 3 : 2);
                        const int kpar = (int)((Qi >> jc) & 1ull) ^ 1;   // parent level parity; D = 2k + 1
                        tab = MAZE_TAB_OPEN | (code << MAZE_TAB_CODE_SHIFT) | ((2 * kpar + 1) << MAZE_TAB_D4_SHIFT);
                        gv = 1;
                    }
                } else if (c & 1) {                              // passage between (i, j) and (i + 1, j)
                    const int j = (c - 1) >> 1;
                    if ((Si >> j) & 1ull) {
                        const bool child_lower = ((P0n >> j) & 1ull) && !((P1n >> j) & 1ull);   // its parent is above
                        const int far = (int)(((child_lower ? Fn : Fi) >> j) & 1ull);
                        const int code = far ? (r < gr ? 0 : 1) : (child_lower ? 1 : 0);
                        const int kpar = (int)(((child_lower ? Qn : Qi) >> j) & 1ull) ^ 1;
                        tab = MAZE_TAB_OPEN | (code << MAZE_TAB_CODE_SHIFT) | ((2 * kpar + 1) << MAZE_TAB_D4_SHIFT);
                        gv = 1;
                    }
                }
            }
            table[r * W + c] = (uint8_t)tab;
            if (grid) grid[r * W + c] = (uint8_t)gv;
        }
    }
}

// Border-less (toroidal) maze: the block grid of the bordered maze without its outer ring
// (lib/maze_generation.py:53-55), written from the register planes; pitch W = Wb - 2.
__device__ __forceinline__ void write_stripped_grid(const Walls& w, int Hb, int Wb, int gi, int gj, uint8_t* __restrict__ grid) {
    const int lane = lane_id();
    const int W = Wb - 2;
    for (int r = 1; r < Hb - 1; ++r) {
        const bool cell_row = (r & 1) != 0;
        const int i = cell_row ? (r - 1) >> 1 : (r >> 1) - 1;
        const u64 Ei = cell_row ? row_get(w.e, i) : 0ull, Si = cell_row ? 0ull : row_get(w.s, i);
        for (int c = 1 + lane; c < Wb - 1; c += 32) {
            int gv = 0;
            if (cell_row) {
                if (c & 1) gv = (i == gi && ((c - 1) >> 1) == gj) ? 2 : 1;
                else gv = (int)((Ei >> ((c - 2) >> 1)) & 1ull);
            } else if (c & 1) {
                gv = (int)((Si >> ((c - 1) >> 1)) & 1ull);
            }
            grid[(r - 1) * W + (c - 1)] = (uint8_t)gv;
        }
    }
}

// ---- warp-per-maze kernel (unscored) ----------------------------------------------------------

__global__ void __launch_bounds__(WARP_GEN_THREADS, 4)
maze_generate_warp_kernel(GenParams p) {
    const int lane = lane_id();
    const int n = p.count_dev ? min(*p.count_dev, p.n) : p.n;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(p.work_counter, 1);
        item = __shfl_sync(FULL, item, 0);
        if (item >= n) break;
        const int m = p.ids ? p.ids[item] : item;
        int32_t* mm = p.meta + (size_t)m * MAZE_META_WORDS;
        const int H = mm[MAZE_META_H], W = mm[MAZE_META_W];
        const int flags = mm[MAZE_META_FLAGS];
        const bool tor = (flags & MAZE_FLAG_TOROIDAL) != 0;
        if (tor && !p.grids) continue;   // without a grid buffer the CTA kernel does the toroidal slots
        const int gen_count = mm[MAZE_META_SPARE];
        const int Hb = tor ? H + 2 : H, Wb = tor ? W + 2 : W;   // :48 gen_maze(shape + 2)
        const int nr = (Hb - 1) / 2, nc = (Wb - 1) / 2;
        if (nr > MAZE_GEN_MAX_CELLS || nc > MAZE_GEN_MAX_CELLS || nr < 1 || nc < 1) {
            if (lane == 0) mm[MAZE_META_SOL_LEN] = -1;
            continue;
        }
        Walls w;
        int si, sj;
        generate_walls(w, (flags >> 8) & 0xff, nr, nc, p.seed,
                       (u64)(p.slot_id_base + m) | ((u64)(unsigned)gen_count << 40), (unsigned)p.candidate_base, si, sj);
        const int goal = select_goal(w, si, sj);
        const int gi = goal >> 8, gj = goal & 0xff;
        if (tor) {   // grid + start / goal now, fields by maze_fields_toroidal_kernel (block-level BFS on the torus)
            write_stripped_grid(w, Hb, Wb, gi, gj, p.grids + (size_t)m * p.slot);
            __syncwarp();
            if (lane == 0) {
                mm[MAZE_META_START] = (2 * si) | ((2 * sj) << 16);
                mm[MAZE_META_GOAL] = (2 * gi) | ((2 * gj) << 16);
                mm[MAZE_META_SOL_LEN] = 0;   // pending: written by the fields kernel
                mm[MAZE_META_SPARE] = gen_count + 1;
            }
            continue;
        }
        GoalField g;
        goal_field(w, gi, gj, si, sj, 2 * (H < W ? H : W), g);
        encode_bordered(w, g, H, W, gi, gj, p.table + (size_t)m * p.slot, p.grids ? p.grids + (size_t)m * p.slot : nullptr);
        __syncwarp();
        if (lane == 0) {
            const int sol_len = 2 * g.start_level + 1;
            mm[MAZE_META_START] = (2 * si + 1) | ((2 * sj + 1) << 16);
            mm[MAZE_META_GOAL] = (2 * gi + 1) | ((2 * gj + 1) << 16);
            mm[MAZE_META_SOL_LEN] = sol_len;
            mm[MAZE_META_MAX_STEPS] = max_steps_budget(H, W, sol_len);
            mm[MAZE_META_SPARE] = gen_count + 1;
        }
    }
}

// ---- scored bulk generation, first half: every (slot, candidate) pair is one work item of the warp generator
// (32 warps per SM hide the dependent-issue latency of carving, which a 4-warp CTA cannot); the walls go to
// scratch as bit-planes (1 KB per candidate), the CTA kernel then only scores and keeps.
__global__ void __launch_bounds__(WARP_GEN_THREADS, 4)
maze_generate_planes_kernel(GenParams p) {
    const int lane = lane_id();
    const int total = p.n * p.candidates;
    for (;;) {
        int work = 0;
        if (lane == 0) work = atomicAdd(p.work_counter, 1);
        work = __shfl_sync(FULL, work, 0);
        if (work >= total) break;
        const int item = work / p.candidates, cand = work - item * p.candidates;
        const int m = p.ids ? p.ids[item] : p.item_base + item;
        const int32_t* mm = p.meta + (size_t)m * MAZE_META_WORDS;
        const int H = mm[MAZE_META_H], W = mm[MAZE_META_W], flags = mm[MAZE_META_FLAGS];
        const bool tor = (flags & MAZE_FLAG_TOROIDAL) != 0;
        const int Hb = tor ? H + 2 : H, Wb = tor ? W + 2 : W;
        const int nr = (Hb - 1) / 2, nc = (Wb - 1) / 2;
        if (nr > MAZE_GEN_MAX_CELLS || nc > MAZE_GEN_MAX_CELLS || nr < 1 || nc < 1) continue;   // the CTA kernel reports it
        Walls w;
        int si, sj;
        generate_walls(w, (flags >> 8) & 0xff, nr, nc, p.seed,
                       (u64)(p.slot_id_base + m) | ((u64)(unsigned)mm[MAZE_META_SPARE] << 40), (unsigned)(p.candidate_base + cand), si, sj);
        const int goal = select_goal(w, si, sj);
        unsigned long long* out = p.planes + (size_t)work * PLANE_WORDS;
        out[lane] = w.e.a0; out[32 + lane] = w.e.a1;
        out[MAZE_GEN_MAX_CELLS + lane] = w.s.a0; out[MAZE_GEN_MAX_CELLS + 32 + lane] = w.s.a1;
        if (lane == 0) {
            out[2 * MAZE_GEN_MAX_CELLS] = (unsigned long long)(unsigned)((si << 8) | sj);
            out[2 * MAZE_GEN_MAX_CELLS + 1] = (unsigned long long)(unsigned)goal;
        }
    }
}

// second half of unscored toroidal generation: fields of the toroidal slots among the items
__global__ void __launch_bounds__(FIELD_THREADS)
maze_fields_toroidal_kernel(GenParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int n = p.count_dev ? min(*p.count_dev, p.n) : p.n;
    FieldSmem f = field_smem_carve(smem, p.smem_hw);
    for (int item = blockIdx.x; item < n; item += gridDim.x) {
        const int m = p.ids ? p.ids[item] : item;
        const int32_t* mm = p.meta + (size_t)m * MAZE_META_WORDS;
        if (!(mm[MAZE_META_FLAGS] & MAZE_FLAG_TOROIDAL) || mm[MAZE_META_SOL_LEN] == -1) continue;
        fields_of_slot(f, p.grids, p.meta, p.table, m, p.slot);
    }
}

// ---- CTA-per-maze kernel (toroidal and / or scored) -------------------------------------------

// block grid bytes of the bordered maze from the wall planes (warp 0)
__device__ __forceinline__ void expand_walls(const Walls& w, uint8_t* grid, int Wb, int nr, int nc) {
    const int lane = lane_id();
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
        const int i = lane + 32 * sl;
        if (i >= nr) continue;
        const u64 e = sl ? w.e.a1 : w.e.a0, s = sl ? w.s.a1 : w.s.a0;
        uint8_t* row = grid + (2 * i + 1) * Wb;
        for (int j = 0; j < nc; ++j) {
            row[2 * j + 1] = 1;
            if ((e >> j) & 1ull) row[2 * j + 2] = 1;
            if ((s >> j) & 1ull) row[Wb + 2 * j + 1] = 1;
        }
    }
}

template <bool kScored>   // kScored: candidates > 1 or a difficulty output (keeps the raw path lean)
__global__ void __launch_bounds__(GEN_THREADS)
maze_generate_kernel(GenParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_start, s_goal, s_keep_start, s_keep_goal, s_take;
    __shared__ double s_keep_diff;
    __shared__ MazeMetrics s_metrics;
    const int tid = threadIdx.x;
    const int n = p.count_dev ? min(*p.count_dev, p.n) : p.n;
    FieldSmem f = field_smem_carve(smem, p.smem_hw);
    const size_t keep_bytes = ((size_t)p.smem_hw + 15) & ~(size_t)15;
    uint8_t* keep = smem + field_smem_bytes(p.smem_hw);
    MetricsSmem ms = metrics_smem_carve(keep + keep_bytes, p.smem_cells, f.queue);

    for (int item = blockIdx.x; item < n; item += gridDim.x) {
        const int m = p.ids ? p.ids[item] : p.item_base + item;
        int32_t* mm = p.meta + (size_t)m * MAZE_META_WORDS;
        const int H = mm[MAZE_META_H], W = mm[MAZE_META_W];
        const int flags = mm[MAZE_META_FLAGS];
        const bool tor = (flags & MAZE_FLAG_TOROIDAL) != 0;
        if (p.only_toroidal && !tor) continue;
        const int algo = (flags >> 8) & 0xff;
        const int gen_count = mm[MAZE_META_SPARE];
        const int Hb = tor ? H + 2 : H, Wb = tor ? W + 2 : W;   // :48 gen_maze(shape + 2)
        const int nr = (Hb - 1) / 2, nc = (Wb - 1) / 2;
        if (nr > MAZE_GEN_MAX_CELLS || nc > MAZE_GEN_MAX_CELLS || nr < 1 || nc < 1 || Hb * Wb > p.smem_hw) {
            if (tid == 0) mm[MAZE_META_SOL_LEN] = -1;
            continue;
        }

        // Candidates are DRAWN four at a time, one per warp (the carving loop is a dependent chain that
        // leaves a lone warp mostly idle), and SCORED one after the other in candidate order by the CTA.
        constexpr int NW = GEN_THREADS / 32;
        const int wid = tid >> 5;
        for (int base = 0; base < p.candidates; base += NW) {
            Walls w;
            int si = 0, sj = 0, goal = 0;
            if (base + wid < p.candidates) {
                if (p.planes) {   // drawn by maze_generate_planes_kernel
                    const unsigned long long* in = p.planes + ((size_t)item * p.candidates + base + wid) * PLANE_WORDS;
                    const int lane = tid & 31;
                    w.e.a0 = in[lane]; w.e.a1 = in[32 + lane];
                    w.s.a0 = in[MAZE_GEN_MAX_CELLS + lane]; w.s.a1 = in[MAZE_GEN_MAX_CELLS + 32 + lane];
                    const int sij = (int)in[2 * MAZE_GEN_MAX_CELLS];
                    si = sij >> 8; sj = sij & 0xff;
                    goal = (int)in[2 * MAZE_GEN_MAX_CELLS + 1];
                } else {
                    generate_walls(w, algo, nr, nc, p.seed, (u64)(p.slot_id_base + m) | ((u64)(unsigned)gen_count << 40),
                                   (unsigned)(p.candidate_base + base + wid), si, sj);
                    goal = select_goal(w, si, sj);
                }
            }
            for (int k = 0; k < NW && base + k < p.candidates; ++k) {
                const int cand = base + k;
                __syncthreads();   // previous item / candidate fully consumed before smem is reused
                for (int i = tid; i < Hb * Wb; i += GEN_THREADS) {
                    f.grid[i] = 0;
                    if (kScored) f.dist[i] = DIST_INF;
                }
                __syncthreads();
                if (wid == k) {
                    expand_walls(w, f.grid, Wb, nr, nc);
                    if ((tid & 31) == 0) {
                        s_start = (2 * si + 1) * Wb + 2 * sj + 1;
                        s_goal = (2 * (goal >> 8) + 1) * Wb + 2 * (goal & 0xff) + 1;
                    }
                    __syncwarp();
                    if ((tid & 31) == 0) f.grid[s_goal] = 2;   // :33
                    if (kScored) cell_bfs_distances(w, si, sj, f.dist, Wb);   // block distances from start for the metrics
                }
                __syncthreads();
                if constexpr (kScored) {
                    // McClendon difficulty of the bordered maze (base_maze_env.py:86-92; for border-less
                    // mazes lib/maze_generation.py:51), on block distances from start
                    maze_metrics(f, ms, Hb, Wb, s_start, s_goal, s_metrics, false);
                    if (tid == 0) {
                        // first wins ties: the double-atomic sums leave equal scores a few ulp apart, in an order that
                        // depends on the maze and may vary run to run, so a later candidate must be lower by > 1e-12
                        s_take = (cand == 0) || (s_metrics.difficulty < s_keep_diff - 1e-12 * fabs(s_keep_diff));
                        if (s_take) { s_keep_diff = s_metrics.difficulty; s_keep_start = s_start; s_keep_goal = s_goal; }
                    }
                    __syncthreads();
                    if (p.candidates > 1 && s_take)
                        for (int i = tid; i < Hb * Wb; i += GEN_THREADS) keep[i] = f.grid[i];
                }
            }
        }
        if (kScored && p.candidates > 1) {
            __syncthreads();
            for (int i = tid; i < Hb * Wb; i += GEN_THREADS) f.grid[i] = keep[i];
            if (tid == 0) { s_start = s_keep_start; s_goal = s_keep_goal; }
            __syncthreads();
        }
        const int start_idx = s_start;
        int sr = start_idx / Wb, sc = start_idx % Wb, gr = s_goal / Wb, gc = s_goal % Wb;

        if (tor) {   // :53-55 strip the outer ring
            uint8_t* tmp = reinterpret_cast<uint8_t*>(f.dist);
            for (int i = tid; i < H * W; i += GEN_THREADS) tmp[i] = f.grid[(i / W + 1) * Wb + (i % W) + 1];
            __syncthreads();
            for (int i = tid; i < H * W; i += GEN_THREADS) f.grid[i] = tmp[i];
            __syncthreads();
            sr -= 1; sc -= 1; gr -= 1; gc -= 1;
        }

        block_bfs(f, H, W, tor, gr * W + gc);
        encode_step_table(f, H, W, tor, gr, gc, p.table + (size_t)m * p.slot);
        if (p.grids) {
            uint8_t* g = p.grids + (size_t)m * p.slot;
            for (int i = tid; i < H * W; i += GEN_THREADS) g[i] = f.grid[i];
        }
        if (tid == 0) {
            const int d = f.dist[sr * W + sc];
            const int sol_len = d == DIST_INF ? 0 : d + 1;
            mm[MAZE_META_START] = sr | (sc << 16);
            mm[MAZE_META_GOAL] = gr | (gc << 16);
            mm[MAZE_META_SOL_LEN] = sol_len;
            mm[MAZE_META_MAX_STEPS] = max_steps_budget(H, W, sol_len);
            mm[MAZE_META_SPARE] = gen_count + 1;
            if (kScored && p.difficulty) p.difficulty[item] = s_keep_diff;
        }
    }
}

}  // namespace

extern "C" int maze_generate(maze_ctx* ctx, uint8_t* grids, int32_t* meta, uint8_t* table, const int32_t* ids,
                             const int32_t* count_dev, int n, int slot, int max_h, int max_w,
                             uint64_t seed, int64_t slot_id_base, int candidates, double* difficulty, void* stream) {
    if (!ctx) return MAZE_E_NULL;
    if (!meta || !table) return maze_fail_arg(ctx, MAZE_E_NULL, "maze_generate pointer");
    if (n <= 0 || slot <= 0) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_generate n / slot");
    if (candidates < 1 || candidates > 64) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_generate candidates (1..64)");
    if (max_h < 5 || max_w < 5 || !(max_h & 1) || !(max_w & 1) || max_h + 2 > MAZE_GEN_MAX_DIM || max_w + 2 > MAZE_GEN_MAX_DIM)
        return maze_fail_arg(ctx, MAZE_E_SHAPE, "maze_generate: max shape must be odd, >= 5 and <= MAZE_GEN_MAX_DIM - 2");
    if (max_h * max_w > slot) return maze_fail_arg(ctx, MAZE_E_RANGE, "maze_generate: slot smaller than max shape");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int sms = ctx->num_sms > 0 ? ctx->num_sms : 148;
    GenParams p;
    p.grids = grids; p.meta = meta; p.table = table; p.ids = ids; p.count_dev = count_dev;
    p.n = n; p.slot = slot;
    p.smem_hw = (max_h + 2) * (max_w + 2);
    const bool scored = candidates > 1 || difficulty != nullptr;
    p.smem_cells = scored ? ((max_h + 1) / 2) * ((max_w + 1) / 2) : 0;
    p.candidates = candidates;
    // Test hook: draw candidates b .. b + k - 1 of every slot instead of 0 .. k - 1, so that a test can materialise each
    // candidate of a best-of-k selection on its own (candidates = 1) and re-score it with the oracle.
    const char* cb = getenv("MAZE_GEN_CANDIDATE_BASE");
    p.candidate_base = cb ? atoi(cb) : 0;
    p.only_toroidal = scored ? 0 : 1;
    p.difficulty = difficulty;
    p.work_counter = nullptr;
    p.seed = seed; p.slot_id_base = slot_id_base;
    p.planes = nullptr; p.item_base = 0;

    if (!scored) {   // bordered slots: one warp per maze, persistent over the items
        int per_sm = 0;
        MAZE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, maze_generate_warp_kernel, WARP_GEN_THREADS, 0));
        if (per_sm < 1) per_sm = 1;
        const int warps_per_cta = WARP_GEN_THREADS / 32;
        const int want = (n + warps_per_cta - 1) / warps_per_cta;
        const int grid = want < per_sm * sms ? want : per_sm * sms;
        p.work_counter = ctx->d_counter;
        MAZE_CHECK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(int), st));
        maze_generate_warp_kernel<<<grid, WARP_GEN_THREADS, 0, st>>>(p);
        MAZE_CHECK(cudaGetLastError());
    }
    if (!scored && grids) {   // toroidal slots: their fields need a block-resolution BFS; CTAs find no work otherwise
        const size_t fsmem = field_smem_bytes(p.smem_hw);
        MAZE_CHECK(cudaFuncSetAttribute(maze_fields_toroidal_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
        int per = 0;
        MAZE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, maze_fields_toroidal_kernel, FIELD_THREADS, fsmem));
        if (per < 1) per = 1;
        maze_fields_toroidal_kernel<<<n < per * sms ? n : per * sms, FIELD_THREADS, fsmem, st>>>(p);
        MAZE_CHECK(cudaGetLastError());
        return 0;
    }
    // scored generation (and toroidal slots when there is no grid buffer): one CTA per maze
    size_t smem = field_smem_bytes(p.smem_hw);
    if (scored) smem += (((size_t)p.smem_hw + 15) & ~(size_t)15) + metrics_smem_bytes(p.smem_cells);
    auto kernel = scored ? maze_generate_kernel<true> : maze_generate_kernel<false>;
    MAZE_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    MAZE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GEN_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    const int resident = per_sm * sms;
    // Bulk best-of-k (host-side n, more than a handful of slots): the candidates are drawn by the warp generator
    // into library-owned scratch, chunk by chunk, and the CTA kernel only scores and keeps.  Regeneration queues
    // (device-side count, a few slots per step) stay on the single-kernel path.
    constexpr int CHUNK = 8192;
    if (scored && candidates > 1 && !count_dev && n >= 16 && !getenv("MAZE_GEN_SINGLE_KERNEL")) {
        const int chunk = n < CHUNK ? n : CHUNK;
        const size_t need = (size_t)chunk * candidates * PLANE_WORDS * sizeof(unsigned long long);
        if (ctx->scratch_bytes < need) {
            MAZE_CHECK(cudaStreamSynchronize(st));
            cudaFree(ctx->d_scratch);
            ctx->d_scratch = nullptr; ctx->scratch_bytes = 0;
            MAZE_CHECK(cudaMalloc(&ctx->d_scratch, need));
            ctx->scratch_bytes = need;
        }
        int wper = 0;
        MAZE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&wper, maze_generate_planes_kernel, WARP_GEN_THREADS, 0));
        if (wper < 1) wper = 1;
        for (int c0 = 0; c0 < n; c0 += chunk) {
            GenParams q = p;
            q.n = n - c0 < chunk ? n - c0 : chunk;
            q.ids = ids ? ids + c0 : nullptr;
            q.item_base = c0;
            q.difficulty = difficulty ? difficulty + c0 : nullptr;
            q.planes = static_cast<unsigned long long*>(ctx->d_scratch);
            q.work_counter = ctx->d_counter;
            MAZE_CHECK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(int), st));
            const int want = (q.n * candidates + WARP_GEN_THREADS / 32 - 1) / (WARP_GEN_THREADS / 32);
            maze_generate_planes_kernel<<<want < wper * sms ? want : wper * sms, WARP_GEN_THREADS, 0, st>>>(q);
            kernel<<<q.n < resident ? q.n : resident, GEN_THREADS, smem, st>>>(q);
        }
        MAZE_CHECK(cudaGetLastError());
        return 0;
    }
    kernel<<<n < resident ? n : resident, GEN_THREADS, smem, st>>>(p);
    MAZE_CHECK(cudaGetLastError());
    return 0;
}
