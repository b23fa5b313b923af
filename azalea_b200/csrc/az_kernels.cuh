// az_kernels.cuh -- the per-move kernels of the search hot path (sm_100a).
//
//   k_select         mcts.select_batch + deduplicate_leaves   (mcts.py:46-152)
//   k_expand_backup  evaluate_batch tail + expand + backup    (mcts.py:192-255)
//   az_reroot        SearchTree.move / reset                  (search_tree.py:59-132)
//   k_play_commit    Policy.choose_action tail + execute_action + play_game
//
// Node record (16 B, one 128-bit access per child):
//   x = num_visits f32, y = total_value f32 (child's own view), z = prior f32,
//   w = link u32: AZ_UNEVAL, or first_child << 9 | num_children (0 = terminal)
// Children of a node are contiguous and in legal-move order, so the k
// children of a node are one coalesced 16*k-byte read by the game's warp
// (lane j%32 holds child j).  `parent` is not stored: the warp keeps the
// path it just walked (node | tile << 23 per level) and backs up along it.
//
// All float arithmetic that decides a move uses the explicitly rounded
// intrinsics (__fadd_rn, __fmul_rn, __fdiv_rn, __fsqrt_rn): one IEEE
// rounding per operation and no FMA contraction, like NumPy float32.
#pragma once

#include "az_common.cuh"

struct az_select_args {
    int batch;
    float coef;
    double noise_scale, noise_alpha;
    int root_mode;      // 1: evaluate_root's selection (mcts.py:18-24)
};

struct az_expand_args {
    int batch;
    int prior_kind;
    const float *value;     // [G][B]
    const float *prior;     // [G][B][nn]
    int root_mode;          // 1: expand the root, no backup (mcts.py:25-26)
};

// ------------------------------------------------------------- leaf output

// Network-view board cells (mcts.py:176-181, hex.py:72-87): cell v of the
// view is tile v of the board (colour 0 to move) or the colour-swapped
// anti-diagonal mirror (colour 1 to move); `rot` turns that view by 180
// degrees (az_engine_set_reflect): cell v reads tile rot(flip?(v)).  Each lane
// packs 4 cells into one 32-bit store; the two masks are staged in shared
// memory so that every lane can test arbitrary tiles.
__device__ __forceinline__ void az_emit_board(const az_engine &e, uint32_t *smask,
                                              uint32_t x, uint32_t o, int flip,
                                              int rot, int8_t *dst)
{
    const int lane = az_lane();
    __syncwarp();
    if (lane < e.NW) { smask[lane] = x; smask[32 + lane] = o; }
    __syncwarp();
    for (int base = 0; base < e.cell_stride; base += 128) {
        int v0 = base + lane * 4;
        uint32_t packed = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            int v = v0 + q;
            uint32_t cell = 0;
            if (v < e.nn) {
                const int vr = rot ? az_rot_tile(v, e.nn) : v;
                int t = flip ? az_flip_tile(vr, e.n, e.div_magic) : vr;
                uint32_t bx = (smask[t >> 5] >> (t & 31)) & 1u;
                uint32_t bo = (smask[32 + (t >> 5)] >> (t & 31)) & 1u;
                // colour swap under flip: X(1) <-> O(2)  (hex.py:84)
                cell = flip ? (bo * 1u + bx * 2u) : (bx * 1u + bo * 2u);
            }
            packed |= cell << (8 * q);
        }
        if (v0 < e.cell_stride)
            *reinterpret_cast<uint32_t *>(dst + v0) = packed;
    }
}

// One orientation coin per network row (az_engine_set_reflect) for descent b of
// the launch, from the game's Philox key and counter (descent, ply): the same
// for any window, stream count, graph or world size.  Everything is re-read
// from meta here so that nothing stays live across k_select's descent loop.
__device__ __forceinline__ int az_reflect_coin(const az_engine &e, const int32_t *meta, int b,
                                               uint32_t domain)
{
    const uint2 key = make_uint2((uint32_t)e.cfg.seed ^ (uint32_t)meta[M_GID_LO],
                                 (uint32_t)(e.cfg.seed >> 32) ^ (uint32_t)meta[M_GID_HI]);
    const uint4 c = make_uint4((uint32_t)(meta[M_SIM] + b), 0u, (uint32_t)meta[M_PLY], domain);
    return (int)(az_philox7(c, key).x & 1u);
}

// ------------------------------------------------------------- root noise

// eta ~ Dirichlet(alpha) over k children, lane j%32 slot j/32 (mcts.py:126-127:
// rng.dirichlet(np.full(k, alpha)); statistical parity, not bit parity).
// eta = g / sum(g) with g ~ Gamma(alpha) by Ahrens-Dieter GS (exact for
// alpha <= 1; larger alpha adds floor(alpha) exponentials), kept in logs
// (base 2: one MUFU per log / exp) because alpha = 0.03 puts most samples far
// below FLT_MIN before normalisation.  Counter-based: (simulation, child, ply)
// -> Philox4x32-7; one block serves the first attempt of the two children
// lane + 32 s and lane + 32 (s + 1) (x, y | z, w), straight-line.  GS rejects
// 3.4 % of its candidates at alpha = 0.03, i.e. about four of a warp's 121
// children per simulation: the rejected ones go round a small loop whose
// uniforms come from a counter hash of (key, simulation, child, ply, attempt)
// -- a full Philox block per retry was most of the generator's cost.
__device__ __forceinline__ float az_lg2(float x)
{
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float az_ex2(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float az_u01f(uint32_t r)    // (0,1), one FMA
{
    return __fmaf_rn((float)(r >> 8), 1.0f / 16777216.0f, 0.5f / 16777216.0f);
}

// One GS attempt for Gamma(a), a <= 1, from two uniforms: r2 = log2 of the candidate; accepted?
__device__ __forceinline__ bool az_gs_try(uint32_t b1, uint32_t b2, float bgs, float agx,
                                          float inv_alpha, float &r2)
{
    const float pgs = bgs * az_u01f(b1);
    const float l2 = az_lg2(az_u01f(b2));
    if (pgs <= 1.0f) {
        r2 = az_lg2(pgs) * inv_alpha;                   // X = P^(1/alpha)
        return l2 <= -1.44269504f * az_ex2(r2);         // U2 <= exp(-X)
    }
    r2 = az_lg2(-0.69314718f * az_lg2((bgs - pgs) * inv_alpha));    // X = -ln((b - P) / alpha)
    return l2 <= (agx - 1.0f) * r2;                     // U2 <= X^(alpha-1)
}

template <int MAXS>
__device__ __forceinline__ void az_dirichlet_noise(int lane, int k, float alpha, uint32_t sim,
                                                   uint32_t ply, uint2 key, float (&noise)[MAXS])
{
    static_assert(MAXS % 2 == 0, "children are drawn in pairs");
    const float alpha_frac = alpha > 1.0f ? alpha - floorf(alpha) : alpha;
    const float agx = alpha_frac > 0.0f ? alpha_frac : 1.0f;
    const float inv_alpha = 1.0f / agx;
    const float bgs = (2.7182818f + agx) / 2.7182818f;
    float lg[MAXS];
    uint32_t todo = 0;                                  // bit s: child lane + 32 s still has no sample
#pragma unroll
    for (int s = 0; s < MAXS; s += 2) {
        lg[s] = lg[s + 1] = -INFINITY;
        if (32 * s < k) {                               // warp-uniform
            const int j0 = lane + 32 * s;
            const uint4 u = az_philox7(make_uint4(sim, (uint32_t)j0, ply, 0xD1C10000u), key);
            float c;
            if (j0 < k) { if (az_gs_try(u.x, u.y, bgs, agx, inv_alpha, c)) lg[s] = c; else todo |= 1u << s; }
            if (j0 + 32 < k) { if (az_gs_try(u.z, u.w, bgs, agx, inv_alpha, c)) lg[s + 1] = c; else todo |= 2u << s; }
        }
    }
    if (__any_sync(AZ_FULL, todo != 0u)) {
        const uint32_t h0 = key.x ^ (sim * 0x9E3779B9u) ^ (ply * 0xC2B2AE35u) ^ ((uint32_t)lane * 0x85EBCA6Bu);
#pragma unroll 1
        for (uint32_t att = 1; att < 24u && todo != 0u; att++) {
#pragma unroll
            for (int s = 0; s < MAXS; s++) {
                if (!((todo >> s) & 1u)) continue;
                const uint32_t w1 = az_fmix32(h0 + att * 0x27D4EB2Fu + (uint32_t)s * 0x165667B1u);
                const uint32_t w2 = az_fmix32(w1 ^ key.y);
                float c;
                if (az_gs_try(w1, w2, bgs, agx, inv_alpha, c)) { lg[s] = c; todo &= ~(1u << s); }
            }
        }
    }
    if (alpha > 1.0f) {
#pragma unroll
        for (int s = 0; s < MAXS; s++) {
            const int j = lane + 32 * s;
            if (j >= k) continue;
            float tot = (alpha_frac > 0.0f) ? az_ex2(lg[s]) : 0.0f;
            for (int m = 0; m < (int)alpha; m++) {
                const uint4 u = az_philox7(make_uint4(sim, (uint32_t)j, ply, 0xE9000000u + m), key);
                tot -= 0.69314718f * az_lg2(az_u01f(u.x));
            }
            lg[s] = az_lg2(tot);
        }
    }
    float mx = lg[0];
#pragma unroll
    for (int s = 1; s < MAXS; s++) mx = fmaxf(mx, lg[s]);
    asm("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(mx) : "f"(mx));
    float z = 0.0f;
#pragma unroll
    for (int s = 0; s < MAXS; s++) { lg[s] = az_ex2(lg[s] - mx); z += lg[s]; }
    for (int off = 16; off; off >>= 1) z += __shfl_xor_sync(AZ_FULL, z, off);
    const float invz = 1.0f / z;
#pragma unroll
    for (int s = 0; s < MAXS; s++) noise[s] = lg[s] * invz;
}

// Test aid: draw the root noise vector each game would use for simulation
// `sim` of its current ply into out[g][0..k).
__global__ void k_noise_sample(az_engine e, float alpha, int k, int sim, float *out)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    const uint2 key = make_uint2((uint32_t)e.cfg.seed ^ (uint32_t)meta[M_GID_LO],
                                 (uint32_t)(e.cfg.seed >> 32) ^ (uint32_t)meta[M_GID_HI]);
    float noise[12];
    az_dirichlet_noise<12>(lane, k, alpha, (uint32_t)sim, (uint32_t)meta[M_PLY], key, noise);
#pragma unroll
    for (int s = 0; s < 12; s++)
        if (lane + 32 * s < k) out[(size_t)g * k + lane + 32 * s] = noise[s];
}

// ------------------------------------------------------------------ select

// Register budget of k_select<4>: 7 CTAs of four warps per SM = 72 registers.  4096 games are 27.7
// warps per SM, so 7 CTAs still hold them all in one wave; measured tree-only throughput by
// minimum CTAs per SM (registers): 8 (64) 1.685e8, 7 (72) 1.746e8, 6 (80) 1.53e8, 5 (96) 1.59e8,
// 4 (120, the first setting without spills) 1.69e8 simulations/s.
#ifndef AZ_SELECT_MINBLOCKS
#define AZ_SELECT_MINBLOCKS 7
#endif
template <int MAXS, bool NOISE>
__global__ void __launch_bounds__(AZ_WARPS_PER_CTA * 32, MAXS <= 4 ? AZ_SELECT_MINBLOCKS : 3)
k_select(az_engine e, az_select_args a)
{
    __shared__ uint32_t smask_all[AZ_WARPS_PER_CTA][64];
    const int lane = az_lane();
    const int wib = threadIdx.x >> 5;
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + wib;
    if (g >= e.g1) return;
    uint32_t *smask = smask_all[wib];
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    int4 *info = e.leaf_info + (size_t)g * e.B;
    const int status = meta[M_STATUS];
    if (status != 0 || meta[M_WINNER] != 0 || meta[M_DRAW] != 0) {
        if (lane < e.B) info[lane] = make_int4(-1, 0, 0, 0);
        return;
    }
    // playout cap: a fast ply's search ends once it has made fast_descents new descents (the
    // unsigned difference: M_SIM is a running counter of the slot)
    if (!a.root_mode && e.fast_descents &&
        (uint32_t)(meta[M_SIM] - meta[M_PLY_SIM0]) >= (uint32_t)e.fast_descents &&
        !az_full_search(e, meta)) {
        if (lane < e.B) info[lane] = make_int4(-1, 0, 0, 0);
        return;
    }
    uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    const uint32_t valid = az_valid_word(lane, e.nn);
    const uint32_t rx = lane < e.NW ? e.board[((size_t)g * 2 + 0) * e.NW + lane] : 0u;
    const uint32_t ro = lane < e.NW ? e.board[((size_t)g * 2 + 1) * e.NW + lane] : 0u;
    const int rcolor = meta[M_COLOR];
    const uint32_t rootlink = nodes[0].w;
    uint32_t *lmask = e.leaf_masks + (size_t)g * e.B * 2 * e.NW;
    int8_t *lboard = e.leaf_board + (size_t)g * e.B * e.cell_stride;

    if (a.root_mode) {
        // every lockstep move starts here: the playout cap counts this move's new descents from
        // this point, tree reuse or not
        if (e.fast_descents && lane == 0) meta[M_PLY_SIM0] = meta[M_SIM];
        // evaluate_root (mcts.py:18-24): the root position itself is the leaf
        if (lane < e.B && lane > 0) info[lane] = make_int4(-1, 0, 0, 0);
        if (rootlink != AZ_UNEVAL) {
            if (lane == 0) info[0] = make_int4(-1, 0, 0, 0);
            return;
        }
        int k = az_count_bits(~(rx | ro) & valid);
        const int coin = e.reflect ? az_reflect_coin(e, meta, 0, AZ_REFLECT_ROOT_DOMAIN) : 0;
        if (lane < e.NW) { lmask[lane] = rx; lmask[e.NW + lane] = ro; }
        az_emit_board(e, smask, rx, ro, rcolor == 2, coin, lboard);
        if (lane == 0) {
            info[0] = make_int4(0, ((rcolor - 1) << 8) | (coin << AZ_LEAF_REFLECTED_BIT), k, 0);
            if (coin) e.counters[(size_t)g * AZ_CNT_PER_GAME + AZ_CNT_REFLECTED_ROWS] += 1;
        }
        return;
    }
    if (rootlink == AZ_UNEVAL || (rootlink & AZ_LINK_KMASK) == 0u) {
        // search_forward asserts an evaluated, non-terminal root
        // (search_tree.py:146-149)
        if (lane == 0) meta[M_STATUS] = status | AZ_ST_ILLEGAL;
        if (lane < e.B) info[lane] = make_int4(-1, 0, 0, 0);
        return;
    }

    // slots beyond this batch must not look like leaves to k_expand_backup,
    // which walks all max_batch slots
    if (lane >= a.batch && lane < e.B) info[lane] = make_int4(-1, 0, 0, 0);
    uint32_t *pathg = e.path + (size_t)g * e.B * e.path_stride;
    const uint2 key = make_uint2((uint32_t)e.cfg.seed ^ (uint32_t)meta[M_GID_LO],
                                 (uint32_t)(e.cfg.seed >> 32) ^ (uint32_t)meta[M_GID_HI]);
    const int sim0 = meta[M_SIM];
    const int ply = meta[M_PLY];
    int my_leaf = -1, my_depth = 0;         // lane b remembers descent b: depth | needs the network << 16 | flip << 17
                                            // | rotated << 18
    const bool pack = (e.cfg.flags & AZ_CFG_PACK_LEAVES) != 0;
    // per launch: small.  nn_rows counts rotated rows (az_engine_set_reflect) in its high half
    uint32_t sum_k = 0, sum_d = 0, uniq = 0, nn_rows = 0, term = 0;

    for (int b = 0; b < a.batch; b++) {
        uint32_t x = rx, o = ro, link = rootlink;
        int color = rcolor, node = 0, depth = 0, tile = 0;
        uint32_t *path = pathg + (size_t)b * e.path_stride;
        // select_leaf, mcts.py:95-116
        while (link != AZ_UNEVAL && (link & AZ_LINK_KMASK) != 0u) {
            const int k = (int)(link & AZ_LINK_KMASK), fc = (int)(link >> AZ_LINK_KBITS);
            uint4 rec[MAXS];
            int ni = 0;
#pragma unroll
            for (int s = 0; s < MAXS; s++) {
                int j = lane + 32 * s;
                rec[s] = j < k ? nodes[fc + j] : make_uint4(0, 0, 0, 0);
                ni += (int)__uint_as_float(rec[s].x);
            }
            // score_actions, mcts.py:119-136.  sum(N) is a sum of small
            // integers: exact in any order.
            const int sum_n = __reduce_add_sync(AZ_FULL, ni);
            const float sq = __fsqrt_rn((float)sum_n);
            const bool sq_zero = sum_n == 0;
            // (drawn after the record loads have been issued: the generator hides their latency;
            // a fast ply of the playout cap draws and mixes none, warp-uniformly)
            float noise[MAXS];
            const bool mix = NOISE && depth == 0 && az_full_search(e, meta);
            if (mix)
                az_dirichlet_noise<MAXS>(lane, k, (float)a.noise_alpha, (uint32_t)(sim0 + b),
                                         (uint32_t)ply, key, noise);
            // forced playouts (az_engine_set_forced_playouts): at the root of a full ply a child
            // with 0 < N < sqrt(k P sum N) scores +inf; warp-uniform, like mix
            const bool force = e.forced_k != 0.0f &&
                               (NOISE ? mix : depth == 0 && az_full_search(e, meta));
            uint32_t bestkey = 0;
            int bestj = 0x7fffffff;
            // sum N == 0 (first descent into a freshly expanded node): every
            // score is (c*P)*0 = +0, and np.argmax takes child 0 whatever the
            // priors are (SURVEY appendix A.2) -- nothing to compute.
            if (sq_zero) {
                bestj = lane == 0 ? 0 : 0x7fffffff;
            } else {
#pragma unroll
            for (int s = 0; s < MAXS; s++) {
                const int j = lane + 32 * s;
                const float nv = __uint_as_float(rec[s].x), tv = __uint_as_float(rec[s].y);
                float pr = __uint_as_float(rec[s].z);
                if (mix)                    // mcts.py:128-131, mixed in float64
                    pr = (float)((1.0 - a.noise_scale) * (double)pr +
                                 a.noise_scale * (double)noise[s]);
                const float cp = __fmul_rn(a.coef, pr);
                float score;
                // Warp-uniform shortcut: if none of these 32 children has been
                // visited, N = W = 0 for all of them, so Q = -0/1 and the visit
                // gap is sqrt(sum N)/1: no division needed.  Most nodes below the
                // root are in this state for most of their slots.
                if (__any_sync(AZ_FULL, nv != 0.0f)) {
                    // A zero numerator sends the IEEE division down its slow
                    // subroutine (FCHK).  0/x = +-0 and (+-0) + u == u for
                    // u >= +0, so those quotients are replaced by an exact 0
                    // without changing a bit of the score.
                    const float gap = __fdiv_rn(sq, __fadd_rn(1.0f, nv));
                    const bool tv_zero = tv == 0.0f;
                    float q = __fdiv_rn(tv_zero ? 1.0f : -tv, fmaxf(nv, 1.0f));
                    q = tv_zero ? 0.0f : q;
                    score = __fadd_rn(q, __fmul_rn(cp, gap));
                    // (an unvisited child is never forced: the other branch needs no test)
                    if (force && nv > 0.0f &&
                        nv < az_forced_visits(e.forced_k, __uint_as_float(rec[s].z), (float)sum_n))
                        score = INFINITY;
                } else {
                    score = __fmul_rn(cp, sq);
                }
                if (j < k) {
                    // + 0.0f folds -0 into +0 so the integer key orders like floats
                    const uint32_t sk = az_orderable(__fadd_rn(score, 0.0f));
                    if (bestj == 0x7fffffff || sk > bestkey) { bestkey = sk; bestj = j; }
                }
            }
            }
            // np.argmax: the lowest index among equal maxima (mcts.py:112)
            const uint32_t mxkey = __reduce_max_sync(AZ_FULL, bestkey);
            const int jstar = __reduce_min_sync(AZ_FULL, (bestj != 0x7fffffff && bestkey == mxkey)
                                                             ? bestj : 0x7fffffff);
            const int owner = jstar & 31, slot = jstar >> 5;
            uint32_t cl = 0, cn = 0, cw = 0;
#pragma unroll
            for (int s = 0; s < MAXS; s++)
                if (s == slot) { cl = rec[s].w; cn = rec[s].x; cw = rec[s].y; }
            const uint32_t clink = __shfl_sync(AZ_FULL, cl, owner);
            node = fc + jstar;
            // virtual loss on the way down (mcts.py:69,79-92): N += 1, W += 1
            // on every node of the path except the root
            if (lane == owner)
                *reinterpret_cast<float2 *>(&nodes[node]) =
                    make_float2(__fadd_rn(__uint_as_float(cn), 1.0f), __fadd_rn(__uint_as_float(cw), 1.0f));
            // ForwardSearchIterator.step, search_tree.py:298-308
            tile = az_kth_empty(~(x | o) & valid, jstar, e.NW);
            if (lane == (tile >> 5)) {
                if (color == 1) x |= 1u << (tile & 31); else o |= 1u << (tile & 31);
            }
            color = 3 - color;
            if (lane == 0) path[depth] = (uint32_t)node | ((uint32_t)tile << 23);
            depth++;
            link = clink;
            sum_k += k;
        }
        sum_d += depth;
        // deduplicate_leaves: first occurrence wins (mcts.py:139-152)
        const bool dup = __any_sync(AZ_FULL, lane < b && my_leaf == node);
        if (lane == b) { my_leaf = node; my_depth = depth; }    // (bits 16, 17 are set below)
        if (dup) {
            if (lane == 0) info[b] = make_int4(-1, 0, 0, depth);
            continue;
        }
        uniq++;
        int flags = 0, kk = 0, coin = 0;
        if (link != AZ_UNEVAL) {
            flags = AZ_LEAF_TERMINAL_KNOWN;
            term++;
        } else {
            const int mover = 3 - color;    // who just played `tile`
            if (az_hex_wins(mover == 1 ? x : o, e.n, e.div_magic, tile, mover)) {
                flags = AZ_LEAF_TERMINAL_NEW;
                term++;
            } else {
                kk = az_count_bits(~(x | o) & valid);
                if (e.reflect) coin = az_reflect_coin(e, meta, b, AZ_REFLECT_DOMAIN);
                // packed leaves: the board is written once the batch's rows have been reserved
                if (!pack) az_emit_board(e, smask, x, o, color == 2, coin, lboard + (size_t)b * e.cell_stride);
                else if (lane == b) my_depth |= (1 << 16) | ((color == 2) << 17) | (coin << 18);
                nn_rows += 1u + ((uint32_t)coin << 16);
            }
            if (lane < e.NW) {
                lmask[(size_t)b * 2 * e.NW + lane] = x;
                lmask[(size_t)b * 2 * e.NW + e.NW + lane] = o;
            }
        }
        if (lane == 0) info[b] = make_int4(node, flags | ((color - 1) << 8) | (coin << AZ_LEAF_REFLECTED_BIT),
                                           kk, depth);
    }
    __syncwarp();
    if (pack) {
        // AZ_CFG_PACK_LEAVES: the leaves the network must evaluate (unique, not terminal:
        // mcts.py:75,192-200) of all games of the window go to consecutive rows -- one
        // reservation per game and batch, then the boards from the masks kept per leaf
        const uint32_t nnmask = __ballot_sync(AZ_FULL, (my_depth >> 16) & 1);
        int row = 0;
        if (lane == 0 && nnmask) row = atomicAdd(&e.leaf_rows[e.g0], __popc(nnmask));
        row = __shfl_sync(AZ_FULL, row, 0);
        const int cap = (e.g1 - e.g0) * e.B;        // rows of the window (a batch cannot exceed it)
        for (uint32_t m = nnmask; m; m &= m - 1, row++) {
            const int b = __ffs(m) - 1;
            const int meta_b = __shfl_sync(AZ_FULL, my_depth, b);
            const int r = row < cap ? row : cap - 1;
            const uint32_t lx = lane < e.NW ? lmask[(size_t)b * 2 * e.NW + lane] : 0u;
            const uint32_t lo = lane < e.NW ? lmask[(size_t)b * 2 * e.NW + e.NW + lane] : 0u;
            az_emit_board(e, smask, lx, lo, (meta_b >> 17) & 1, (meta_b >> 18) & 1,
                          e.leaf_board + ((size_t)e.g0 * e.B + r) * e.cell_stride);
            if (lane == 0) info[b].w = (meta_b & 0xffff) | (r << 10);
        }
        my_depth &= 0xffff;
    }
    // undo the virtual losses, leaf list order (mcts.py:72)
    for (int b = 0; b < a.batch; b++) {
        const int depth = __shfl_sync(AZ_FULL, my_depth, b);
        const uint32_t *path = pathg + (size_t)b * e.path_stride;
        for (int dd = lane; dd < depth; dd += 32) {
            float2 *p = reinterpret_cast<float2 *>(&nodes[path[dd] & AZ_MAX_NODE]);
            float2 nw = *p;
            nw.x = __fadd_rn(nw.x, -1.0f);
            nw.y = __fadd_rn(nw.y, -1.0f);
            *p = nw;
        }
        __syncwarp();
    }
    if (lane == 0) {
        meta[M_SIM] = sim0 + a.batch;
        unsigned long long *cnt = e.counters + (size_t)g * AZ_CNT_PER_GAME;
        cnt[AZ_CNT_SIMULATIONS] += a.batch;
        cnt[AZ_CNT_SUM_CHILDREN] += sum_k;
        cnt[AZ_CNT_SUM_DEPTH] += sum_d;
        cnt[AZ_CNT_UNIQUE_LEAVES] += uniq;
        cnt[AZ_CNT_NN_ROWS] += nn_rows & 0xffffu;
        cnt[AZ_CNT_TERMINAL_LEAVES] += term;
        if (nn_rows >> 16) cnt[AZ_CNT_REFLECTED_ROWS] += nn_rows >> 16;
    }
}

// ---------------------------------------------------------- expand + backup

template <int MAXS>
__global__ void __launch_bounds__(AZ_WARPS_PER_CTA * 32)
k_expand_backup(az_engine e, az_expand_args a)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    // packed leaves: the evaluator has consumed this window's batch; the next az_mcts_select
    // starts a new one
    const bool pack = (e.cfg.flags & AZ_CFG_PACK_LEAVES) != 0 && !a.root_mode;
    if (pack && g == e.g0 && lane == 0) e.leaf_rows[e.g0] = 0;
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    int status = meta[M_STATUS];
    if (status != 0) return;
    uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    const int4 *info = e.leaf_info + (size_t)g * e.B;
    const uint32_t *pathg = e.path + (size_t)g * e.B * e.path_stride;
    const uint32_t *lmask = e.leaf_masks + (size_t)g * e.B * 2 * e.NW;
    const uint32_t valid = az_valid_word(lane, e.nn);
    int tail = meta[M_TAIL];
    long long vref = ((long long)(uint32_t)meta[M_VREF_LO]) | ((long long)meta[M_VREF_HI] << 32);
    unsigned long long expanded = 0, skipped = 0;
    const bool soft_full = (e.cfg.flags & AZ_CFG_SOFT_POOL_FULL) != 0;

    for (int b = 0; b < a.batch; b++) {
        const int4 inf = info[b];
        if (inf.x < 0) continue;
        const int node = inf.x, flags = inf.y & 0xff, lcolor = (inf.y >> 8) & 1;
        const int lrot = (inf.y >> AZ_LEAF_REFLECTED_BIT) & 1;
        const int k = inf.z, depth = pack ? (inf.w & 1023) : inf.w;
        const size_t row = pack ? (size_t)e.g0 * e.B + (size_t)(inf.w >> 10) : (size_t)g * e.B + b;
        // evaluate_batch, mcts.py:192-200: terminal positions are worth -1
        // to the player to move
        const float v = flags ? -1.0f : a.value[row];
        bool expand = !(flags & AZ_LEAF_TERMINAL_KNOWN);
        if (expand) {
            // create_child_nodes, search_tree.py:254-274
            if (vref + k > e.cfg.max_nodes_ref) { status |= AZ_ST_TREE_FULL; break; }
            if (tail + k > e.C || tail + k > AZ_MAX_NODE) {
                // this half of the game's pool is exhausted (no reference analogue: its pool
                // is MAX_NODES).  Soft mode: the leaf stays unevaluated -- its value is still
                // backed up below, and a later visit expands it once the next re-root has
                // compacted the pool; otherwise the game is flagged and dropped.
                if (!soft_full) { status |= AZ_ST_POOL_FULL; break; }
                expand = false;
                skipped++;
            }
        }
        if (expand) {
            const int fc = tail;
            if (k > 0) {
                const float *prow = a.prior + row * e.nn;
                if (a.prior_kind == AZ_PRIOR_PROBS) {
                    for (int j = lane; j < k; j += 32)
                        nodes[fc + j] = make_uint4(0u, 0u, __float_as_uint(prow[j]), AZ_UNEVAL);
                } else {
                    // policy head tail (network.py:146-151) + mcts.py:210:
                    // gather the legal tiles' logits, log-softmax, exp.
                    // Lane owns tiles 32*s + lane; the ordinal of an empty
                    // tile is the number of empty tiles before it.  A row the
                    // network saw rotated holds the logit of view tile u at
                    // n*n-1-u; the lane still owns the true tile, so the
                    // reductions below run in the same order either way.
                    const uint32_t occ = lane < e.NW
                        ? (lmask[(size_t)b * 2 * e.NW + lane] | lmask[(size_t)b * 2 * e.NW + e.NW + lane]) : ~0u;
                    const uint32_t emp = ~occ & valid;
                    float lg[MAXS], mx = -INFINITY;
                    int ord[MAXS], base = 0;
#pragma unroll
                    for (int s = 0; s < MAXS; s++) {
                        uint32_t es = __shfl_sync(AZ_FULL, emp, s);
                        ord[s] = -1;
                        lg[s] = -INFINITY;
                        if ((es >> lane) & 1u) {
                            int t = 32 * s + lane;
                            ord[s] = base + __popc(es & ((1u << lane) - 1u));
                            const int u = lcolor ? az_flip_tile(t, e.n, e.div_magic) : t;
                            lg[s] = prow[lrot ? az_rot_tile(u, e.nn) : u];
                            mx = fmaxf(mx, lg[s]);
                        }
                        base += __popc(es);
                    }
                    for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(AZ_FULL, mx, off));
                    float z = 0.0f;
#pragma unroll
                    for (int s = 0; s < MAXS; s++) if (ord[s] >= 0) z += expf(lg[s] - mx);
                    for (int off = 16; off; off >>= 1) z += __shfl_xor_sync(AZ_FULL, z, off);
                    const float logz = logf(z);
#pragma unroll
                    for (int s = 0; s < MAXS; s++)
                        if (ord[s] >= 0)
                            nodes[fc + ord[s]] = make_uint4(0u, 0u,
                                __float_as_uint(expf(lg[s] - mx - logz)), AZ_UNEVAL);
                }
            }
            if (lane == 0) nodes[node].w = ((uint32_t)fc << AZ_LINK_KBITS) | (uint32_t)k;
            tail += k;
            vref += k;
            expanded += k;
        }
        if (!a.root_mode) {
            // backup_batch, mcts.py:242-255: leaf .. root inclusive, the value
            // changes sign at every level.  Path nodes are distinct, so the
            // lanes update them independently; leaves go in list order.
            const uint32_t *path = pathg + (size_t)b * e.path_stride;
            for (int dd = lane; dd < depth; dd += 32) {
                float2 *p = reinterpret_cast<float2 *>(&nodes[path[dd] & AZ_MAX_NODE]);
                float2 nw = *p;
                nw.x = __fadd_rn(nw.x, 1.0f);
                nw.y = __fadd_rn(nw.y, ((depth - 1 - dd) & 1) ? -v : v);
                *p = nw;
            }
            if (lane == 31) {
                float2 *p = reinterpret_cast<float2 *>(&nodes[0]);
                float2 nw = *p;
                nw.x = __fadd_rn(nw.x, 1.0f);
                nw.y = __fadd_rn(nw.y, (depth & 1) ? -v : v);
                *p = nw;
            }
        }
        __syncwarp();
    }
    if (lane == 0) {
        meta[M_TAIL] = tail;
        meta[M_VREF_LO] = (int32_t)(uint32_t)(vref & 0xffffffffll);
        meta[M_VREF_HI] = (int32_t)(vref >> 32);
        meta[M_STATUS] = status;
        e.counters[(size_t)g * AZ_CNT_PER_GAME + AZ_CNT_EXPANDED_CHILDREN] += expanded;
        if (skipped) e.counters[(size_t)g * AZ_CNT_PER_GAME + AZ_CNT_POOL_SKIPPED] += skipped;
    }
}

// ---------------------------------------------------------------- re-root

__device__ __forceinline__ void az_tree_reset(uint4 *nodes, int32_t *meta, int lane)
{
    // SearchTree.reset, search_tree.py:59-71
    if (lane == 0) {
        nodes[0] = make_uint4(0u, 0u, __float_as_uint(1.0f), AZ_UNEVAL);
        meta[M_TAIL] = 1;
        meta[M_VREF_LO] = 1;
        meta[M_VREF_HI] = 0;
    }
}

// SearchTree.move, search_tree.py:115-132.  The reference only moves root_id
// and never frees memory; here the kept subtree is copied breadth-first into
// the other half of the game's pool (new root = node 0), so a game's pool
// stays bounded by one move's growth plus what it keeps.  Visit counts,
// values and priors are carried over unchanged.
__device__ __forceinline__ void az_reroot(const az_engine &e, int g, int32_t *meta,
                                          int move_id, int lane)
{
    const int half = meta[M_HALF];
    uint4 *src = e.nodes + ((size_t)g * 2 + half) * e.C;
    uint4 *dst = e.nodes + ((size_t)g * 2 + (half ^ 1)) * e.C;
    const uint32_t rootlink = src[0].w;
    if (rootlink == AZ_UNEVAL) { az_tree_reset(src, meta, lane); return; }
    const int k0 = (int)(rootlink & AZ_LINK_KMASK);
    if (move_id < 0 || move_id >= k0) {
        if (lane == 0) meta[M_STATUS] |= AZ_ST_ILLEGAL;
        return;
    }
    const uint4 child = src[(rootlink >> AZ_LINK_KBITS) + move_id];
    if (child.w == AZ_UNEVAL) { az_tree_reset(src, meta, lane); return; }
    __syncwarp();
    if (lane == 0) dst[0] = child;
    __syncwarp();
    int head = 0, tail = 1;
    while (head < tail) {
        // 32 queued nodes at a time: their child blocks get consecutive ranges
        const int i = head + lane;
        uint32_t link = i < tail ? dst[i].w : AZ_UNEVAL;
        int k = link == AZ_UNEVAL ? 0 : (int)(link & AZ_LINK_KMASK);
        int incl = k;
        for (int off = 1; off < 32; off <<= 1) {
            int t = __shfl_up_sync(AZ_FULL, incl, off);
            if (lane >= off) incl += t;
        }
        const int nfc = tail + incl - k;
        if (k > 0) dst[i].w = ((uint32_t)nfc << AZ_LINK_KBITS) | (uint32_t)k;
        const int total = __shfl_sync(AZ_FULL, incl, 31);
        for (int q = 0; q < 32; q++) {
            const int kq = __shfl_sync(AZ_FULL, k, q);
            if (kq == 0) continue;
            const int ofc = (int)(__shfl_sync(AZ_FULL, link, q) >> AZ_LINK_KBITS);
            const int dfc = __shfl_sync(AZ_FULL, nfc, q);
            for (int j = lane; j < kq; j += 32) dst[dfc + j] = src[ofc + j];
        }
        __syncwarp();
        head += 32;
        if (head > tail) head = tail;
        tail += total;
    }
    if (lane == 0) {
        meta[M_HALF] = half ^ 1;
        meta[M_TAIL] = tail;
        e.counters[(size_t)g * AZ_CNT_PER_GAME + AZ_CNT_COMPACTED_NODES] += tail;
    }
}
