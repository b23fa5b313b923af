// az_engine.cu -- C ABI (include/azalea_b200.h) + game / lockstep-play kernels.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared
//        -Xcompiler -fPIC   (see __graft_entry__.build()).
// No torch, no CPU fallback: every entry point launches sm_100a kernels.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "az_kernels.cuh"
#include "az_nn_glue.cuh"
#include "az_tower.cuh"
#include "az_block.cuh"

static thread_local char g_cuda_err[256] = "";

static int az_check(cudaError_t err)
{
    if (err == cudaSuccess) return AZ_OK;
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(err),
             cudaGetErrorString(err));
    return AZ_E_CUDA;
}

// Kernels launch on the CURRENT device; an engine (and the stream the caller passes) belongs to
// e->device.  Make that device current for the duration of the call when it is not already.
struct az_device_guard {
    int prev, changed;
    explicit az_device_guard(int dev) : prev(dev), changed(0)
    {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
    }
    ~az_device_guard() { if (changed) cudaSetDevice(prev); }
};

#define AZ_MAX_DEVICES 64

// per-device facts for the engine-less evaluator kernels (they run on the current device)
static int az_current_device()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return dev < 0 || dev >= AZ_MAX_DEVICES ? 0 : dev;
}

static int az_sm_count(int dev)
{
    static int cache[AZ_MAX_DEVICES];       // 0 = unknown; racing writers store the same value
    if (cache[dev] == 0) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        cache[dev] = n > 0 ? n : 148;
    }
    return cache[dev];
}

static inline int az_grid(const az_engine *e)
{
    return (e->g1 - e->g0 + AZ_WARPS_PER_CTA - 1) / AZ_WARPS_PER_CTA;
}

#define AZ_LAUNCH(kernel, e, stream, ...)                                              \
    do {                                                                               \
        az_device_guard guard_((e)->device);                                           \
        kernel<<<az_grid(e), AZ_WARPS_PER_CTA * 32, 0, (cudaStream_t)(stream)>>>(*(e), \
                                                                      ##__VA_ARGS__); \
        return az_check(cudaGetLastError());                                           \
    } while (0)

// ------------------------------------------------------------ game kernels

__device__ __forceinline__ void az_game_reset(const az_engine &e, int g, int32_t *meta,
                                              int lane, bool new_id)
{
    // HexGame.reset (hex.py:47-49) + Policy.reset (policy.py:72-76)
    if (lane < e.NW) {
        e.board[((size_t)g * 2 + 0) * e.NW + lane] = 0u;
        e.board[((size_t)g * 2 + 1) * e.NW + lane] = 0u;
    }
    uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    az_tree_reset(nodes, meta, lane);
    // resignation: no value seen yet by either colour of the new game
    if (lane < 2) e.resign[(size_t)g * AZ_RESIGN_INTS + AZ_RS_MIN + lane] = 0x7f800000u;    // +inf
    if (lane == 0) {
        meta[M_COLOR] = 1;
        meta[M_WINNER] = 0;
        meta[M_PLY] = 0;
        meta[M_STATUS] = 0;
        meta[M_DRAW] = 0;
        meta[M_LAST] = -1;
        if (new_id) {
            long long gid = ((long long)(uint32_t)meta[M_GID_LO]) | ((long long)meta[M_GID_HI] << 32);
            gid += e.cfg.game_id_stride;
            meta[M_GID_LO] = (int32_t)(uint32_t)(gid & 0xffffffffll);
            meta[M_GID_HI] = (int32_t)(gid >> 32);
            meta[M_SERIAL] += 1;
        }
    }
}

__global__ void k_reset(az_engine e, const uint8_t *mask, int init)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    if (mask && !mask[g]) return;
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    if (init) {
        if (lane < AZ_META_INTS) meta[lane] = 0;
        if (lane < AZ_CNT_PER_GAME) e.counters[(size_t)g * AZ_CNT_PER_GAME + lane] = 0ull;
        for (int i = lane; i < AZ_RESIGN_INTS; i += 32) e.resign[(size_t)g * AZ_RESIGN_INTS + i] = 0u;
        if (g == 0 && lane < 16) e.globals[lane] = 0ull;
        __syncwarp();
        if (lane == 0) {
            long long gid = e.cfg.first_game_id + g;
            meta[M_GID_LO] = (int32_t)(uint32_t)(gid & 0xffffffffll);
            meta[M_GID_HI] = (int32_t)(gid >> 32);
        }
        __syncwarp();
    }
    az_game_reset(e, g, meta, lane, false);
}

// HexGameImpl.step on the root position (hex.py:172-179)
__device__ __forceinline__ int az_root_step(const az_engine &e, int g, int32_t *meta,
                                            int tile, int lane)
{
    uint32_t *bx = e.board + ((size_t)g * 2 + 0) * e.NW;
    uint32_t *bo = e.board + ((size_t)g * 2 + 1) * e.NW;
    uint32_t x = lane < e.NW ? bx[lane] : 0u, o = lane < e.NW ? bo[lane] : 0u;
    const int color = meta[M_COLOR];
    const uint32_t bit = 1u << (tile & 31);
    const bool taken = __any_sync(AZ_FULL, lane == (tile >> 5) && ((x | o) & bit));
    if (tile < 0 || tile >= e.nn || taken || meta[M_WINNER] != 0) {
        if (lane == 0) meta[M_STATUS] |= AZ_ST_ILLEGAL;     // hex.py:174-176
        return -1;
    }
    if (lane == (tile >> 5)) {
        if (color == 1) { x |= bit; bx[lane] = x; } else { o |= bit; bo[lane] = o; }
    }
    const bool won = az_hex_wins(color == 1 ? x : o, e.n, e.div_magic, tile, color);
    if (lane == 0) {
        meta[M_COLOR] = 3 - color;
        meta[M_WINNER] = won ? color : 0;
        meta[M_PLY] += 1;
        meta[M_LAST] = tile;
    }
    return won ? color : 0;
}

__global__ void k_hex_step(az_engine e, const int32_t *moves, int32_t *results)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    const int move = moves[g];
    int winner = meta[M_WINNER];
    if (move != 0) {
        int w = az_root_step(e, g, meta, move - 1, lane);
        if (w >= 0) winner = w;
    }
    // HexGameImpl.result, hex.py:161-170
    if (results && lane == 0) results[g] = winner == 0 ? 0 : (winner == 2 ? 1 : 3);
}

__global__ void k_hex_state(az_engine e, int8_t *board, int32_t *color, int32_t *result,
                            int32_t *ply)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    if (board) {
        const uint32_t *bx = e.board + ((size_t)g * 2 + 0) * e.NW;
        const uint32_t *bo = e.board + ((size_t)g * 2 + 1) * e.NW;
        for (int t = lane; t < e.nn; t += 32) {
            uint32_t x = (bx[t >> 5] >> (t & 31)) & 1u, o = (bo[t >> 5] >> (t & 31)) & 1u;
            board[(size_t)g * e.nn + t] = (int8_t)(x + 2u * o);
        }
    }
    if (lane == 0) {
        const int w = meta[M_WINNER];
        if (color) color[g] = meta[M_COLOR] - 1;
        if (result) result[g] = meta[M_DRAW] ? 2 : (w == 0 ? 0 : (w == 2 ? 1 : 3));
        if (ply) ply[g] = meta[M_PLY];
    }
}

__global__ void k_hex_legal(az_engine e, int32_t *moves, int32_t *count)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    const uint32_t valid = az_valid_word(lane, e.nn);
    uint32_t occ = lane < e.NW
        ? (e.board[((size_t)g * 2 + 0) * e.NW + lane] | e.board[((size_t)g * 2 + 1) * e.NW + lane]) : ~0u;
    // hex.py:152-153: no legal moves once the game is won
    uint32_t emp = meta[M_WINNER] ? 0u : (~occ & valid);
    int base = 0;
    int32_t *row = moves + (size_t)g * e.nn;
    for (int s = 0; s < e.NW; s++) {
        uint32_t es = __shfl_sync(AZ_FULL, emp, s);
        if ((es >> lane) & 1u)
            row[base + __popc(es & ((1u << lane) - 1u))] = 32 * s + lane + 1;
        base += __popc(es);
    }
    for (int j = base + lane; j < e.nn; j += 32) row[j] = 0;
    if (count && lane == 0) count[g] = base;
}

__global__ void k_hex_set_state(az_engine e, const int8_t *board, const int32_t *color,
                                const int32_t *last_tile, int reset_trees)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    uint32_t x = 0, o = 0;
    for (int s = 0; s < e.NW; s++) {
        int t = 32 * s + lane;
        int8_t c = t < e.nn ? board[(size_t)g * e.nn + t] : 0;
        uint32_t wx = __ballot_sync(AZ_FULL, c == 1), wo = __ballot_sync(AZ_FULL, c == 2);
        if (lane == s) { x = wx; o = wo; }
    }
    if (lane < e.NW) {
        e.board[((size_t)g * 2 + 0) * e.NW + lane] = x;
        e.board[((size_t)g * 2 + 1) * e.NW + lane] = o;
    }
    const int ply = az_count_bits(x | o);
    if (reset_trees) {
        uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
        az_tree_reset(nodes, meta, lane);
    }
    int winner = 0;
    const int lt = last_tile ? last_tile[g] : -1;
    if (lt >= 0 && lt < e.nn) {
        const bool isx = __any_sync(AZ_FULL, lane == (lt >> 5) && ((x >> (lt & 31)) & 1u));
        const bool iso = __any_sync(AZ_FULL, lane == (lt >> 5) && ((o >> (lt & 31)) & 1u));
        if (isx && az_hex_wins(x, e.n, e.div_magic, lt, 1)) winner = 1;
        if (iso && az_hex_wins(o, e.n, e.div_magic, lt, 2)) winner = 2;
    }
    if (lane == 0) {
        meta[M_COLOR] = color[g];
        meta[M_WINNER] = winner;
        meta[M_PLY] = ply;
        meta[M_STATUS] = 0;
        meta[M_DRAW] = 0;
        meta[M_LAST] = lt;
    }
}

// network-view legal moves of the current leaves (prep.py:15-21 padding,
// hex.py:105-121 flip): original ascending tile order, flipped coordinates
__global__ void k_leaf_moves(az_engine e)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const uint32_t valid = az_valid_word(lane, e.nn);
    for (int b = 0; b < e.B; b++) {
        const int4 inf = e.leaf_info[(size_t)g * e.B + b];
        int32_t *row = e.leaf_moves + ((size_t)g * e.B + b) * e.nn;
        int base = 0;
        if (inf.x >= 0 && (inf.y & 0xff) == 0) {
            const uint32_t *lm = e.leaf_masks + ((size_t)g * e.B + b) * 2 * e.NW;
            const int flip = (inf.y >> 8) & 1;
            uint32_t emp = lane < e.NW ? (~(lm[lane] | lm[e.NW + lane]) & valid) : 0u;
            for (int s = 0; s < e.NW; s++) {
                uint32_t es = __shfl_sync(AZ_FULL, emp, s);
                if ((es >> lane) & 1u) {
                    int t = 32 * s + lane;
                    row[base + __popc(es & ((1u << lane) - 1u))] =
                        (flip ? az_flip_tile(t, e.n, e.div_magic) : t) + 1;
                }
                base += __popc(es);
            }
        }
        for (int j = base + lane; j < e.nn; j += 32) row[j] = 0;
    }
}

__global__ void k_root_stats(az_engine e, float *visits, float *total_value, float *prior,
                             int32_t *num_children, float *root_nw, int64_t *num_nodes)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    const uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    const uint4 root = nodes[0];
    int k = -1, fc = 0;
    if (root.w != AZ_UNEVAL) { k = (int)(root.w & AZ_LINK_KMASK); fc = (int)(root.w >> AZ_LINK_KBITS); }
    for (int j = lane; j < e.nn; j += 32) {
        uint4 r = j < k ? nodes[fc + j] : make_uint4(0, 0, 0, 0);
        if (visits) visits[(size_t)g * e.nn + j] = __uint_as_float(r.x);
        if (total_value) total_value[(size_t)g * e.nn + j] = __uint_as_float(r.y);
        if (prior) prior[(size_t)g * e.nn + j] = __uint_as_float(r.z);
    }
    if (lane == 0) {
        if (num_children) num_children[g] = k;
        if (root_nw) {
            root_nw[2 * g] = __uint_as_float(root.x);
            root_nw[2 * g + 1] = __uint_as_float(root.y);
        }
        if (num_nodes)
            num_nodes[g] = ((long long)(uint32_t)meta[M_VREF_LO]) | ((long long)meta[M_VREF_HI] << 32);
    }
}

// RandomPolicy.choose_action (random_policy.py:25-41) in terms of the tree: one
// visit on every child of the (expanded) root, so that az_play_commit with
// temperature 1 draws the move uniformly and records moves_prob = 1 / k.
__global__ void k_root_uniform(az_engine e)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    if (meta[M_STATUS] != 0) return;
    uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    const uint4 root = nodes[0];
    if (root.w == AZ_UNEVAL) return;
    const int k = (int)(root.w & AZ_LINK_KMASK), fc = (int)(root.w >> AZ_LINK_KBITS);
    for (int j = lane; j < k; j += 32) {
        uint4 r = nodes[fc + j];
        r.x = __float_as_uint(1.0f);
        r.y = 0u;
        nodes[fc + j] = r;
    }
}

__global__ void k_tree_move(az_engine e, const int32_t *move_ids)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const int mv = move_ids[g];
    if (mv < 0) return;
    az_reroot(e, g, e.meta + (size_t)g * AZ_META_INTS, mv, lane);
}

__global__ void k_status(az_engine e, int32_t *status)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.G) status[g] = e.meta[(size_t)g * AZ_META_INTS + M_STATUS];
}

// Deterministic stub evaluator (test / bench aid): same arithmetic as
// oracle/azalea_oracle.c:ostub_eval, on the network view of each leaf.
__global__ void k_stub_eval(az_engine e, int mode)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    const uint32_t valid = az_valid_word(lane, e.nn);
    for (int b = 0; b < e.B; b++) {
        const int4 inf = e.leaf_info[(size_t)g * e.B + b];
        if (inf.x < 0 || (inf.y & 0xff) != 0) continue;
        const uint32_t *lm = e.leaf_masks + ((size_t)g * e.B + b) * 2 * e.NW;
        const int flip = (inf.y >> 8) & 1;
        const uint32_t x = lane < e.NW ? lm[lane] : 0u, o = lane < e.NW ? lm[e.NW + lane] : 0u;
        // board hash: sum over stones of fmix32((2*view_tile + view_colour) * K)
        uint32_t part = 0;
        for (int s = 0; s < e.NW; s++) {
            uint32_t xs = __shfl_sync(AZ_FULL, x, s), os = __shfl_sync(AZ_FULL, o, s);
            int t = 32 * s + lane;
            uint32_t c = ((xs >> lane) & 1u) + 2u * ((os >> lane) & 1u);
            if (c) {
                uint32_t vt = flip ? (uint32_t)az_flip_tile(t, e.n, e.div_magic) : (uint32_t)t;
                uint32_t vc = flip ? 3u - c : c;
                part += az_fmix32((2u * vt + vc) * 0x9E3779B1u);
            }
        }
        const uint32_t h0 = az_fmix32(__reduce_add_sync(AZ_FULL, part) ^ (uint32_t)e.n);
        float value;
        if (mode == 0) value = 0.0f;
        else if (mode == 1) value = __fdiv_rn((float)((int)((h0 >> 8) % 17u) - 8), 8.0f);
        else value = __fadd_rn(__fmul_rn((float)(h0 >> 8), 1.0f / 8388608.0f), -1.0f);
        const size_t row = (size_t)g * e.B + b;
        if (lane == 0) e.value[row] = value;
        // weights by ordinal, prior = w / sum(w) with one IEEE division
        const uint32_t emp = ~(x | o) & valid;
        uint32_t wsum = 0;
        for (int pass = 0; pass < 2; pass++) {
            int base = 0;
            uint32_t wpart = 0;
            for (int s = 0; s < e.NW; s++) {
                uint32_t es = __shfl_sync(AZ_FULL, emp, s);
                if ((es >> lane) & 1u) {
                    int t = 32 * s + lane;
                    uint32_t vt = flip ? (uint32_t)az_flip_tile(t, e.n, e.div_magic) : (uint32_t)t;
                    uint32_t hj = az_fmix32(h0 ^ (vt * 0x9E3779B1u + 0x7F4A7C15u));
                    uint32_t w = mode == 0 ? 1u : (mode == 1 ? 1u + (hj >> 28) : 1u + (hj >> 24));
                    if (pass == 0) wpart += w;
                    else e.prior[row * e.nn + base + __popc(es & ((1u << lane) - 1u))] =
                             __fdiv_rn((float)w, (float)wsum);
                }
                base += __popc(es);
            }
            if (pass == 0) wsum = __reduce_add_sync(AZ_FULL, wpart);
        }
    }
}

// ------------------------------------------------------------ lockstep play

// A game of `nply` plies ended with `result`: flush its history rows to the replay output, count
// it and (auto_reset) start the next game in the slot.
__device__ __forceinline__ void az_finish_game(const az_engine &e, const az_play_params &p, int g,
                                               int32_t *meta, unsigned long long *cnt, int lane,
                                               int nply, int result)
{
    // play_game.py:63-67: reward = result - 2 for the first player's rows,
    // negated on the second player's
    if (p.collect_replay) {
        const int plies = min(nply, e.hist_rows);
        const uint8_t *src = e.hist + (size_t)g * e.hist_rows * e.row_bytes;
        // playout cap: only the rows of full-search plies (reserved bit 0 clear) are flushed
        int rows = plies;
        if (e.fast_descents) {
            int kept = 0;
            for (int r = lane; r < plies; r += 32)
                kept += !(reinterpret_cast<const az_row_header *>(src + (size_t)r * e.row_bytes)->reserved & 1);
            rows = __reduce_add_sync(AZ_FULL, kept);
        }
        // reserve `rows` output rows; the cursor only ever advances by reservations that fit,
        // so concurrent finishers can never be handed space beyond the capacity
        unsigned long long base = ~0ull;
        if (lane == 0) {
            unsigned long long cur = *(volatile unsigned long long *)&e.globals[0];
            for (;;) {
                if (cur + (unsigned long long)rows > (unsigned long long)e.cfg.replay_rows) break;
                const unsigned long long prev = atomicCAS(&e.globals[0], cur, cur + (unsigned long long)rows);
                if (prev == cur) { base = cur; break; }
                cur = prev;
            }
        }
        base = __shfl_sync(AZ_FULL, base, 0);
        if (base != ~0ull) {
            uint8_t *dst = e.replay + (size_t)base * e.row_bytes;
            if (rows == plies) {
                const size_t n16 = (size_t)rows * e.row_bytes / 16;
                for (size_t i = lane; i < n16; i += 32)
                    reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
            } else {
                // the kept rows, compacted in ply order
                const int n16 = e.row_bytes / 16;
                uint8_t *d = dst;
                for (int r = 0; r < plies; r++) {
                    const uint8_t *s = src + (size_t)r * e.row_bytes;
                    if (reinterpret_cast<const az_row_header *>(s)->reserved & 1) continue;
                    for (int i = lane; i < n16; i += 32)
                        reinterpret_cast<uint4 *>(d)[i] = reinterpret_cast<const uint4 *>(s)[i];
                    d += e.row_bytes;
                }
            }
            __syncwarp();
            for (int r = lane; r < rows; r += 32) {
                az_row_header *h = reinterpret_cast<az_row_header *>(dst + (size_t)r * e.row_bytes);
                float rw = (float)(result - 2);
                h->reward = (h->ply & 1) ? -rw : rw;    // the row's own ply (rows may be skipped)
                h->result = result;
                h->game_len = nply;
            }
            if (lane == 0) cnt[AZ_CNT_REPLAY_ROWS] += rows;
        } else if (lane == 0) {
            cnt[AZ_CNT_REPLAY_DROPPED] += rows;
        }
    }
    if (lane == 0) cnt[AZ_CNT_GAMES] += 1;
    __syncwarp();
    if (p.auto_reset) az_game_reset(e, g, meta, lane, true);
}

// Policy target pruning: the PUCT score of a root child {N, W, P, link} as if it had n visits, with
// k_select's operation order and zero shortcut.  Q keeps the child's real N: the paper holds the
// utility estimate constant.
__device__ __forceinline__ float az_prune_score(uint4 c, float sq, float coef, float n)
{
    const float nv = __uint_as_float(c.x), tv = __uint_as_float(c.y);
    const float q = tv == 0.0f ? 0.0f : __fdiv_rn(-tv, fmaxf(nv, 1.0f));
    return __fadd_rn(q, __fmul_rn(__fmul_rn(coef, __uint_as_float(c.z)), __fdiv_rn(sq, __fadd_rn(1.0f, n))));
}

// The pruned count of a visited child other than the most-visited one: the fewest visits n' that
// still score below the most-visited child's s_best, but at least N - floor(n_forced) and at most
// N; one left at 1 becomes 0.  The score falls with n' (every rounding is monotone), so a
// bisection finds the same n' as a scan.
__device__ __forceinline__ float az_pruned_visits(uint4 c, float sq, float sum_n, float s_best,
                                                  float coef, float k)
{
    const float nv = __uint_as_float(c.x);
    const float d = floorf(az_forced_visits(k, __uint_as_float(c.z), sum_n));
    int lo = d >= nv ? 0 : (int)nv - (int)d, hi = (int)nv;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (az_prune_score(c, sq, coef, (float)mid) < s_best) hi = mid; else lo = mid + 1;
    }
    return lo == 1 ? 0.0f : (float)lo;
}

__global__ void __launch_bounds__(AZ_WARPS_PER_CTA * 32)
k_play_commit(az_engine e, az_play_params p, int32_t *chosen)
{
    const int lane = az_lane();
    const int g = e.g0 + blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= e.g1) return;
    int32_t *meta = e.meta + (size_t)g * AZ_META_INTS;
    unsigned long long *cnt = e.counters + (size_t)g * AZ_CNT_PER_GAME;
    const int status = meta[M_STATUS];
    const int ply = meta[M_PLY];
    if (status & AZ_ST_DISABLED) return;
    if (status & AZ_ST_ILLEGAL) return;     // a bug, not a game outcome: keep it visible
    if (status != 0) {
        // SearchTreeFull: the reference drops the game and starts another
        // (parallel_player.py:71-76)
        if (lane == 0) {
            cnt[AZ_CNT_GAMES_FAILED] += 1;
            if (chosen) reinterpret_cast<int4 *>(chosen)[g] = make_int4(0, -1, -1, ply);
        }
        __syncwarp();
        if (p.auto_reset) az_game_reset(e, g, meta, lane, true);
        return;
    }
    if (meta[M_WINNER] != 0 || meta[M_DRAW] != 0) {
        if (chosen && lane == 0) reinterpret_cast<int4 *>(chosen)[g] = make_int4(0, -1, -1, ply);
        return;
    }
    uint4 *nodes = e.nodes + ((size_t)g * 2 + meta[M_HALF]) * e.C;
    const uint32_t rootlink = nodes[0].w;
    if (rootlink == AZ_UNEVAL || (rootlink & AZ_LINK_KMASK) == 0u) {
        if (lane == 0) meta[M_STATUS] = status | AZ_ST_ILLEGAL;
        return;
    }
    const int k = (int)(rootlink & AZ_LINK_KMASK), fc = (int)(rootlink >> AZ_LINK_KBITS);
    const int nslots = (k + 31) >> 5;
    // resignation (az_engine_set_resign), after the search and before the move is drawn:
    // r = max(Q_root, Q_best) for the player to move.  A node's W is from the view of the
    // player to move there, so Q_best = -W/N of the most-visited child (lowest ordinal on ties).
    if (e.resign_on) {
        const int best = az_most_visited(nodes, fc, k, lane);
        const uint4 root = nodes[0];
        float r = __fdiv_rn(__uint_as_float(root.y), __uint_as_float(root.x));
        if (best < k) {
            const uint4 c = nodes[fc + best];
            r = fmaxf(r, -__fdiv_rn(__uint_as_float(c.y), __uint_as_float(c.x)));
        }
        const int color = meta[M_COLOR];
        uint32_t *rs = e.resign + (size_t)g * AZ_RESIGN_INTS;
        if (az_calibration_game(e, meta)) {
            // never resigns: keep each colour's lowest r for the bookkeeping at the game's end
            if (lane == 0)
                rs[AZ_RS_MIN + color - 1] =
                    __float_as_uint(fminf(__uint_as_float(rs[AZ_RS_MIN + color - 1]), r));
        } else if (r < e.resign_thresh) {
            // the mover resigns: no move, no row for this ply, the opponent wins
            const int result = color == 1 ? 1 : 3;
            if (lane == 0) {
                meta[M_WINNER] = 3 - color;
                rs[AZ_RS_RESIGNED] += 1;
                if (chosen) reinterpret_cast<int4 *>(chosen)[g] = make_int4(0, -1, result, ply);
            }
            __syncwarp();
            az_finish_game(e, p, g, meta, cnt, lane, ply, result);
            return;
        }
    }
    // Policy.choose_action, policy.py:142-149
    float temp = 0.0f;
    if (p.move_sampling && ply < p.exploration_depth) temp = p.temperature;
    const uint2 key = make_uint2((uint32_t)e.cfg.seed ^ (uint32_t)meta[M_GID_LO],
                                 (uint32_t)(e.cfg.seed >> 32) ^ (uint32_t)meta[M_GID_HI]);
    const uint4 rnd = az_philox(make_uint4(0u, 0u, (uint32_t)ply, 0xC0111700u), key);

    // as_distribution + multinomial (search_tree.py:327-344, policy.py:160):
    // temperature 0 = uniform over the arg-max ties, otherwise p ~ N^(1/T)
    int move_id = 0;
    if (temp == 0.0f) {
        int mx = 0;
        for (int s = 0; s < nslots; s++) {
            int j = lane + 32 * s;
            int nv = j < k ? (int)__uint_as_float(nodes[fc + j].x) : -1;
            mx = max(mx, __reduce_max_sync(AZ_FULL, nv));
        }
        int ties = 0;
        for (int s = 0; s < nslots; s++) {
            int j = lane + 32 * s;
            bool hit = j < k && (int)__uint_as_float(nodes[fc + j].x) == mx;
            ties += __popc(__ballot_sync(AZ_FULL, hit));
        }
        int pick = (int)(rnd.x % (uint32_t)ties);
        for (int s = 0; s < nslots; s++) {
            int j = lane + 32 * s;
            bool hit = j < k && (int)__uint_as_float(nodes[fc + j].x) == mx;
            uint32_t ball = __ballot_sync(AZ_FULL, hit);
            int c = __popc(ball);
            if (pick < c) { move_id = 32 * s + az_nth_set_bit(ball, pick); break; }
            pick -= c;
        }
    } else {
        double tot = 0.0;
        const double inv_t = 1.0 / (double)temp;
        for (int s = 0; s < nslots; s++) {
            int j = lane + 32 * s;
            double w = 0.0;
            if (j < k) {
                float nv = __uint_as_float(nodes[fc + j].x);
                w = temp == 1.0f ? (double)nv : (nv > 0.0f ? pow((double)nv, inv_t) : 0.0);
            }
            for (int off = 16; off; off >>= 1) w += __shfl_xor_sync(AZ_FULL, w, off);
            tot += w;
        }
        const double target = tot * (((double)rnd.x + 0.5) * (1.0 / 4294967296.0));
        double acc = 0.0;
        move_id = -1;
        for (int s = 0; s < nslots && move_id < 0; s++) {
            int j = lane + 32 * s;
            double w = 0.0;
            if (j < k) {
                float nv = __uint_as_float(nodes[fc + j].x);
                w = temp == 1.0f ? (double)nv : (nv > 0.0f ? pow((double)nv, inv_t) : 0.0);
            }
            double incl = w;
            for (int off = 1; off < 32; off <<= 1) {
                double t = __shfl_up_sync(AZ_FULL, incl, off);
                if (lane >= off) incl += t;
            }
            uint32_t ball = __ballot_sync(AZ_FULL, w > 0.0 && acc + incl > target);
            if (ball) move_id = 32 * s + __ffs(ball) - 1;
            acc += __shfl_sync(AZ_FULL, incl, 31);
        }
        if (move_id < 0) {
            // rounding left target == total: take the last visited child
            for (int s = nslots - 1; s >= 0 && move_id < 0; s--) {
                int j = lane + 32 * s;
                bool hit = j < k && __uint_as_float(nodes[fc + j].x) > 0.0f;
                uint32_t ball = __ballot_sync(AZ_FULL, hit);
                if (ball) move_id = 32 * s + 31 - __clz(ball);
            }
            if (move_id < 0) move_id = 0;
        }
    }

    const uint32_t valid = az_valid_word(lane, e.nn);
    const uint32_t x = lane < e.NW ? e.board[((size_t)g * 2 + 0) * e.NW + lane] : 0u;
    const uint32_t o = lane < e.NW ? e.board[((size_t)g * 2 + 1) * e.NW + lane] : 0u;
    const int tile = az_kth_empty(~(x | o) & valid, move_id, e.NW);
    const int color = meta[M_COLOR];
    // playout cap: this ply had the fast search; its row stays out of the replay output
    const bool fast = !az_full_search(e, meta);

    // replay row before the move (play_game.py:90-96)
    if (p.collect_replay && ply < e.hist_rows) {
        uint8_t *row = e.hist + ((size_t)g * e.hist_rows + ply) * e.row_bytes;
        if (lane == 0) {
            az_row_header h;
            h.game_id = ((long long)(uint32_t)meta[M_GID_LO]) | ((long long)meta[M_GID_HI] << 32);
            h.ply = ply;
            h.color = color - 1;
            h.num_moves = k;
            h.reward = 0.0f;
            h.result = 0;
            h.temperature = temp;
            h.move = tile + 1;
            h.move_id = move_id;
            h.game_len = 0;
            h.reserved = fast ? 1 : 0;      // history rows only: flushed rows keep 0
            *reinterpret_cast<az_row_header *>(row) = h;
        }
        int8_t *cells = reinterpret_cast<int8_t *>(row + sizeof(az_row_header));
        for (int s = 0; s < e.NW; s++) {
            uint32_t xs = __shfl_sync(AZ_FULL, x, s), os = __shfl_sync(AZ_FULL, o, s);
            int t = 32 * s + lane;
            if (t < e.cell_stride) cells[t] = (int8_t)(((xs >> lane) & 1u) + 2u * ((os >> lane) & 1u));
        }
        float *vis = reinterpret_cast<float *>(row + sizeof(az_row_header) + e.cell_stride);
        if (e.forced_k != 0.0f && !fast) {
            // policy target pruning (Wu 2019, section 3.2): the row gets the visits PUCT would
            // have given without forced playouts; the move above was drawn from the raw ones
            const int best = az_most_visited(nodes, fc, k, lane);
            int ni = 0;
            for (int j = lane; j < k; j += 32) ni += (int)__uint_as_float(nodes[fc + j].x);
            const float sum_n = (float)__reduce_add_sync(AZ_FULL, ni);
            const float sq = __fsqrt_rn(sum_n);
            float s_best = 0.0f;
            if (best < k) {
                const uint4 c = nodes[fc + best];
                s_best = az_prune_score(c, sq, e.prune_coef, __uint_as_float(c.x));
            }
            for (int j = lane; j < e.nn; j += 32) {
                float v = 0.0f;
                if (j < k) {
                    const uint4 c = nodes[fc + j];
                    v = __uint_as_float(c.x);
                    if (j != best && v > 0.0f)
                        v = az_pruned_visits(c, sq, sum_n, s_best, e.prune_coef, e.forced_k);
                }
                vis[j] = v;
            }
        } else {
            for (int j = lane; j < e.nn; j += 32)
                vis[j] = j < k ? __uint_as_float(nodes[fc + j].x) : 0.0f;
        }
    }
    __syncwarp();

    // AzaleaAgent.execute_action, azalea_agent.py:60-64: tree first, then game
    az_reroot(e, g, meta, move_id, lane);
    __syncwarp();
    const int won = az_root_step(e, g, meta, tile, lane);
    __syncwarp();
    const int nply = ply + 1;
    int result = won > 0 ? (won == 2 ? 1 : 3) : 0;
    bool over = won > 0;
    if (!over && nply >= e.cfg.max_plies) {
        // play_game.py:57-61: no winner within game_max_length -> draw
        over = true;
        result = 2;
        if (lane == 0) meta[M_DRAW] = 1;
    }
    if (lane == 0) {
        cnt[AZ_CNT_PLIES] += 1;
        if (fast) cnt[AZ_CNT_FAST_PLIES] += 1;
        if (chosen) reinterpret_cast<int4 *>(chosen)[g] = make_int4(tile + 1, move_id, result, nply);
        // a calibration game ended with a winner: would the winner have resigned at some ply?
        if (won > 0 && e.resign_on && az_calibration_game(e, meta)) {
            uint32_t *rs = e.resign + (size_t)g * AZ_RESIGN_INTS;
            const float m = __uint_as_float(rs[AZ_RS_MIN + won - 1]);
            rs[AZ_RS_CALIB] += 1;
            rs[AZ_RS_FALSE_POS] += m < e.resign_thresh ? 1u : 0u;
            const int bin = (int)floorf(__fmul_rn(__fadd_rn(m, 1.0f), 64.0f));
            rs[AZ_RS_HIST + min(AZ_RS_BINS - 1, max(0, bin))] += 1;
        }
    }
    if (!over) return;
    az_finish_game(e, p, g, meta, cnt, lane, nply, result);
}

__global__ void k_replay_clear(az_engine e)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) e.globals[0] = 0ull;
}


// ---------------------------------------------------------- replay collate

// prep.torch_batch_replays (prep.py:24-39) for replay rows that never left
// the device: one warp per sampled row -> padded training tensors.
// pi = as_distribution(visits, temperature) (search_tree.py:327-344) in
// float64, cast to float32.
__global__ void k_replay_collate(const uint8_t *rows, int row_bytes, const int64_t *idx, int count,
                                 int n, int cell_stride, int32_t *board, int32_t *moves,
                                 float *probs, float *reward, int64_t *color, int64_t *result,
                                 int32_t *num_moves)
{
    const int lane = az_lane();
    const int i = blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (i >= count) return;
    const int nn = n * n;
    const uint8_t *row = rows + (size_t)idx[i] * row_bytes;
    const az_row_header h = *reinterpret_cast<const az_row_header *>(row);
    const int8_t *cells = reinterpret_cast<const int8_t *>(row + sizeof(az_row_header));
    const float *vis = reinterpret_cast<const float *>(row + sizeof(az_row_header) + cell_stride);
    const int k = h.num_moves;
    // distribution over the k legal moves
    double tot = 0.0;
    float mx = 0.0f;
    for (int j = lane; j < k; j += 32) mx = fmaxf(mx, vis[j]);
    for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(AZ_FULL, mx, off));
    const double inv_t = h.temperature > 0.0f ? 1.0 / (double)h.temperature : 0.0;
    for (int j = lane; j < k; j += 32) {
        const float v = vis[j];
        double w;
        if (h.temperature > 0.0f) w = v > 0.0f ? (h.temperature == 1.0f ? (double)v : pow((double)v, inv_t)) : 0.0;
        else w = v == mx ? 1.0 : 0.0;
        tot += w;
    }
    for (int off = 16; off; off >>= 1) tot += __shfl_xor_sync(AZ_FULL, tot, off);
    for (int j = lane; j < nn; j += 32) {
        float p = 0.0f;
        if (j < k) {
            const float v = vis[j];
            double w;
            if (h.temperature > 0.0f) w = v > 0.0f ? (h.temperature == 1.0f ? (double)v : pow((double)v, inv_t)) : 0.0;
            else w = v == mx ? 1.0 : 0.0;
            p = (float)(w / tot);
        }
        probs[(size_t)i * nn + j] = p;
    }
    // board and ascending legal moves (hex.py:151-159), zero padded
    int base = 0;
    for (int t0 = 0; t0 < nn; t0 += 32) {
        const int t = t0 + lane;
        const int c = t < nn ? cells[t] : 1;
        if (t < nn) board[(size_t)i * nn + t] = c;
        const uint32_t emp = __ballot_sync(AZ_FULL, c == 0);
        if (c == 0) moves[(size_t)i * nn + base + __popc(emp & ((1u << lane) - 1u))] = t + 1;
        base += __popc(emp);
    }
    for (int j = base + lane; j < nn; j += 32) moves[(size_t)i * nn + j] = 0;
    if (lane == 0) {
        reward[i] = h.reward;
        color[i] = h.color;
        result[i] = 0;          // states are recorded before the move: ongoing
        num_moves[i] = k;
    }
}

// ---------------------------------------------------------- batch reflect

// random_reflect of a collated training batch (the reference's hex.py:124-134
// hook): rows with a coin are turned by 180 degrees, tile t -> n*n-1-t, in
// place.  One warp per row; every element is swapped with its mirror by one
// lane, so the rotation is its own inverse.
__global__ void k_batch_reflect(int32_t *board, int32_t *moves, float *probs, const uint8_t *coins,
                                int count, int nn, int width, int ld)
{
    const int lane = az_lane();
    const int i = blockIdx.x * AZ_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (i >= count || !coins[i]) return;
    int32_t *b = board + (size_t)i * nn;
    for (int t = lane; t < nn / 2; t += 32) {
        const int32_t c = b[t];
        b[t] = b[nn - 1 - t];
        b[nn - 1 - t] = c;
    }
    int32_t *m = moves + (size_t)i * ld;
    float *p = probs + (size_t)i * ld;
    // the legal moves are ascending and zero padded: k = non-zero entries
    int k = 0;
    for (int j0 = 0; j0 < width; j0 += 32) {
        const int j = j0 + lane;
        k += __popc(__ballot_sync(AZ_FULL, j < width && m[j] != 0));
    }
    for (int j = lane; j < (k + 1) / 2; j += 32) {
        const int jr = k - 1 - j;
        const int32_t a = m[j], z = m[jr];
        const float pa = p[j], pz = p[jr];
        m[j] = nn + 1 - z;
        m[jr] = nn + 1 - a;
        p[j] = pz;
        p[jr] = pa;
    }
}

// =================================================================== C ABI

static size_t az_align(size_t x) { return (x + 255) & ~(size_t)255; }

static int az_layout(az_engine *e, const az_config *cfg)
{
    if (!cfg || cfg->num_games < 1 || cfg->board_size < 2 || cfg->board_size > 19 ||
        cfg->max_batch < 1 || cfg->max_batch > 32 || cfg->nodes_per_game < 2 ||
        cfg->nodes_per_game > AZ_MAX_NODE || cfg->replay_rows < 0)
        return AZ_E_INVALID;
    memset(e, 0, sizeof(*e));
    e->cfg = *cfg;
    e->G = cfg->num_games;
    e->g0 = 0;
    e->g1 = e->G;
    e->n = cfg->board_size;
    e->nn = e->n * e->n;
    e->NW = (e->nn + 31) / 32;
    e->B = cfg->max_batch;
    e->C = cfg->nodes_per_game;
    e->cell_stride = (e->nn + 15) & ~15;
    e->path_stride = (e->nn + 3) & ~3;
    e->row_bytes = (int)((sizeof(az_row_header) + e->cell_stride + 4 * (size_t)e->nn + 15) & ~(size_t)15);
    e->hist_rows = cfg->max_plies > 0 && cfg->max_plies < e->nn ? cfg->max_plies : e->nn;
    if (e->cfg.max_plies <= 0) e->cfg.max_plies = 300;
    if (e->cfg.max_nodes_ref <= 0) e->cfg.max_nodes_ref = 10000000;
    if (e->cfg.game_id_stride <= 0) e->cfg.game_id_stride = e->G;
    if (cfg->replay_rows == 0) e->hist_rows = 0;
    e->div_magic = 65536u / (uint32_t)e->n + 1u;
    size_t off = 0;
    size_t o_nodes = off; off = az_align(off + (size_t)e->G * 2 * e->C * sizeof(uint4));
    size_t o_board = off; off = az_align(off + (size_t)e->G * 2 * e->NW * 4);
    size_t o_meta = off; off = az_align(off + (size_t)e->G * AZ_META_INTS * 4);
    size_t o_path = off; off = az_align(off + (size_t)e->G * e->B * e->path_stride * 4);
    size_t o_info = off; off = az_align(off + (size_t)e->G * e->B * sizeof(int4));
    size_t o_lmask = off; off = az_align(off + (size_t)e->G * e->B * 2 * e->NW * 4);
    size_t o_lboard = off; off = az_align(off + (size_t)e->G * e->B * e->cell_stride);
    size_t o_lmoves = off; off = az_align(off + (size_t)e->G * e->B * e->nn * 4);
    size_t o_value = off; off = az_align(off + (size_t)e->G * e->B * 4);
    size_t o_prior = off; off = az_align(off + (size_t)e->G * e->B * e->nn * 4);
    size_t o_cnt = off; off = az_align(off + (size_t)e->G * AZ_CNT_PER_GAME * 8);
    size_t o_glob = off; off = az_align(off + 16 * 8);
    size_t o_lrows = off; off = az_align(off + (size_t)e->G * 4);
    size_t o_hist = off; off = az_align(off + (size_t)e->G * e->hist_rows * e->row_bytes);
    size_t o_replay = off; off = az_align(off + (size_t)e->cfg.replay_rows * e->row_bytes);
    size_t o_resign = off; off = az_align(off + (size_t)e->G * AZ_RESIGN_INTS * 4);
    e->total_bytes = off;
    // offsets are stored as pointers relative to NULL until create() binds them
    e->nodes = (uint4 *)o_nodes;
    e->board = (uint32_t *)o_board;
    e->meta = (int32_t *)o_meta;
    e->path = (uint32_t *)o_path;
    e->leaf_info = (int4 *)o_info;
    e->leaf_masks = (uint32_t *)o_lmask;
    e->leaf_board = (int8_t *)o_lboard;
    e->leaf_moves = (int32_t *)o_lmoves;
    e->value = (float *)o_value;
    e->prior = (float *)o_prior;
    e->counters = (unsigned long long *)o_cnt;
    e->globals = (unsigned long long *)o_glob;
    e->leaf_rows = (int32_t *)o_lrows;
    e->hist = (uint8_t *)o_hist;
    e->replay = (uint8_t *)o_replay;
    e->resign = (uint32_t *)o_resign;
#define AZ_DESC(which, off_, bytes_, elem_, nd_, s0, s1, s2, s3)                         \
    do {                                                                                 \
        az_buffer_desc *d = &e->desc[which];                                             \
        d->offset = off_; d->bytes = bytes_; d->elem_bytes = elem_; d->ndim = nd_;       \
        d->shape[0] = s0; d->shape[1] = s1; d->shape[2] = s2; d->shape[3] = s3;          \
    } while (0)
    AZ_DESC(AZ_BUF_LEAF_BOARD, o_lboard, (size_t)e->G * e->B * e->cell_stride, 1, 3, e->G, e->B, e->cell_stride, 0);
    AZ_DESC(AZ_BUF_LEAF_INFO, o_info, (size_t)e->G * e->B * 16, 4, 3, e->G, e->B, 4, 0);
    AZ_DESC(AZ_BUF_VALUE, o_value, (size_t)e->G * e->B * 4, 4, 2, e->G, e->B, 0, 0);
    AZ_DESC(AZ_BUF_PRIOR, o_prior, (size_t)e->G * e->B * e->nn * 4, 4, 3, e->G, e->B, e->nn, 0);
    AZ_DESC(AZ_BUF_META, o_meta, (size_t)e->G * AZ_META_INTS * 4, 4, 2, e->G, AZ_META_INTS, 0, 0);
    AZ_DESC(AZ_BUF_REPLAY, o_replay, (size_t)e->cfg.replay_rows * e->row_bytes, 1, 2, e->cfg.replay_rows, e->row_bytes, 0, 0);
    AZ_DESC(AZ_BUF_COUNTERS, o_cnt, (size_t)e->G * AZ_CNT_PER_GAME * 8, 8, 2, e->G, AZ_CNT_PER_GAME, 0, 0);
    AZ_DESC(AZ_BUF_LEAF_MOVES, o_lmoves, (size_t)e->G * e->B * e->nn * 4, 4, 3, e->G, e->B, e->nn, 0);
    AZ_DESC(AZ_BUF_GLOBALS, o_glob, 16 * 8, 8, 1, 16, 0, 0, 0);
    AZ_DESC(AZ_BUF_LEAF_ROWS, o_lrows, (size_t)e->G * 4, 4, 1, e->G, 0, 0, 0);
    AZ_DESC(AZ_BUF_RESIGN, o_resign, (size_t)e->G * AZ_RESIGN_INTS * 4, 4, 2, e->G, AZ_RESIGN_INTS, 0, 0);
#undef AZ_DESC
    return AZ_OK;
}

extern "C" {

int az_abi_version(void) { return AZ_ABI_VERSION; }

const char *az_strerror(int code)
{
    switch (code) {
    case AZ_OK: return "ok";
    case AZ_E_INVALID: return "invalid argument";
    case AZ_E_CUDA: return "CUDA error";
    case AZ_E_NOMEM: return "device block too small";
    case AZ_E_UNSUPPORTED: return "unsupported";
    default: return "unknown error";
    }
}

const char *az_last_cuda_error(void) { return g_cuda_err; }

size_t az_engine_device_bytes(const az_config *cfg)
{
    az_engine tmp;
    if (az_layout(&tmp, cfg) != AZ_OK) return 0;
    return tmp.total_bytes;
}

int az_engine_create(az_engine **out, const az_config *cfg, void *mem_dev, size_t mem_bytes,
                     int device)
{
    if (!out || !mem_dev) return AZ_E_INVALID;
    az_engine *e = (az_engine *)calloc(1, sizeof(az_engine));
    if (!e) return AZ_E_INVALID;
    int rc = az_layout(e, cfg);
    if (rc != AZ_OK) { free(e); return rc; }
    if (mem_bytes < e->total_bytes) { free(e); return AZ_E_NOMEM; }
    if (((uintptr_t)mem_dev & 255) != 0) { free(e); return AZ_E_INVALID; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { free(e); return AZ_E_INVALID; }
    az_device_guard guard(device);
    e->device = device;
    char *base = (char *)mem_dev;
#define AZ_BIND(field, type) e->field = (type)(base + (size_t)e->field)
    AZ_BIND(nodes, uint4 *);
    AZ_BIND(board, uint32_t *);
    AZ_BIND(meta, int32_t *);
    AZ_BIND(path, uint32_t *);
    AZ_BIND(leaf_info, int4 *);
    AZ_BIND(leaf_masks, uint32_t *);
    AZ_BIND(leaf_board, int8_t *);
    AZ_BIND(leaf_moves, int32_t *);
    AZ_BIND(value, float *);
    AZ_BIND(prior, float *);
    AZ_BIND(counters, unsigned long long *);
    AZ_BIND(globals, unsigned long long *);
    AZ_BIND(leaf_rows, int32_t *);
    AZ_BIND(hist, uint8_t *);
    AZ_BIND(replay, uint8_t *);
    AZ_BIND(resign, uint32_t *);
#undef AZ_BIND
    // scratch the evaluator reads even for unused slots must be defined
    rc = az_check(cudaMemsetAsync(e->leaf_board, 0, (size_t)e->G * e->B * e->cell_stride, 0));
    // no leaves yet: node = -1 in every slot
    if (rc == AZ_OK) rc = az_check(cudaMemsetAsync(e->leaf_info, 0xff, (size_t)e->G * e->B * sizeof(int4), 0));
    if (rc == AZ_OK) rc = az_check(cudaMemsetAsync(e->meta, 0, (size_t)e->G * AZ_META_INTS * 4, 0));
    if (rc == AZ_OK) rc = az_check(cudaMemsetAsync(e->leaf_rows, 0, (size_t)e->G * 4, 0));
    if (rc == AZ_OK) rc = az_check(cudaMemsetAsync(e->value, 0, (size_t)e->G * e->B * 4, 0));
    if (rc == AZ_OK) rc = az_check(cudaMemsetAsync(e->prior, 0, (size_t)e->G * e->B * e->nn * 4, 0));
    // replay rows carry alignment padding that no kernel writes
    if (rc == AZ_OK && e->hist_rows)
        rc = az_check(cudaMemsetAsync(e->hist, 0, (size_t)e->G * e->hist_rows * e->row_bytes, 0));
    if (rc == AZ_OK && e->cfg.replay_rows)
        rc = az_check(cudaMemsetAsync(e->replay, 0, (size_t)e->cfg.replay_rows * e->row_bytes, 0));
    if (rc == AZ_OK) {
        k_reset<<<az_grid(e), AZ_WARPS_PER_CTA * 32, 0, 0>>>(*e, NULL, 1);
        rc = az_check(cudaGetLastError());
    }
    if (rc == AZ_OK) rc = az_check(cudaStreamSynchronize(0));
    if (rc != AZ_OK) { free(e); return rc; }
    *out = e;
    return AZ_OK;
}

void az_engine_destroy(az_engine *e) { free(e); }

int az_engine_buffer(const az_engine *e, int which, az_buffer_desc *out)
{
    if (!e || !out || which < 0 || which >= AZ_BUF__COUNT) return AZ_E_INVALID;
    *out = e->desc[which];
    return AZ_OK;
}

int az_replay_row_bytes(const az_engine *e) { return e ? e->row_bytes : AZ_E_INVALID; }

int az_games_reset(az_engine *e, const uint8_t *mask_dev, void *stream)
{
    if (!e) return AZ_E_INVALID;
    AZ_LAUNCH(k_reset, e, stream, mask_dev, 0);
}

int az_hex_step(az_engine *e, const int32_t *moves_dev, int32_t *results_dev, void *stream)
{
    if (!e || !moves_dev) return AZ_E_INVALID;
    AZ_LAUNCH(k_hex_step, e, stream, moves_dev, results_dev);
}

int az_hex_state(az_engine *e, int8_t *board_dev, int32_t *color_dev, int32_t *result_dev,
                 int32_t *ply_dev, void *stream)
{
    if (!e) return AZ_E_INVALID;
    AZ_LAUNCH(k_hex_state, e, stream, board_dev, color_dev, result_dev, ply_dev);
}

int az_hex_legal_moves(az_engine *e, int32_t *moves_dev, int32_t *count_dev, void *stream)
{
    if (!e || !moves_dev) return AZ_E_INVALID;
    AZ_LAUNCH(k_hex_legal, e, stream, moves_dev, count_dev);
}

int az_hex_set_state(az_engine *e, const int8_t *board_dev, const int32_t *color_dev,
                     const int32_t *last_tile_dev, int reset_trees, void *stream)
{
    if (!e || !board_dev || !color_dev) return AZ_E_INVALID;
    AZ_LAUNCH(k_hex_set_state, e, stream, board_dev, color_dev, last_tile_dev, reset_trees);
}

static int az_select_launch(az_engine *e, const az_select_args &a, void *stream)
{
    const bool noise = a.noise_scale != 0.0 && !a.root_mode;
    if (e->NW <= 4) {
        if (noise) AZ_LAUNCH((k_select<4, true>), e, stream, a);
        AZ_LAUNCH((k_select<4, false>), e, stream, a);
    } else {
        if (noise) AZ_LAUNCH((k_select<12, true>), e, stream, a);
        AZ_LAUNCH((k_select<12, false>), e, stream, a);
    }
}

int az_mcts_select_root(az_engine *e, void *stream)
{
    if (!e) return AZ_E_INVALID;
    az_select_args a;
    a.batch = 1; a.coef = 0.0f; a.noise_scale = 0.0; a.noise_alpha = 1.0; a.root_mode = 1;
    return az_select_launch(e, a, stream);
}

int az_mcts_select(az_engine *e, const az_search_params *p, void *stream)
{
    if (!e || !p || p->batch_size < 1 || p->batch_size > e->B) return AZ_E_INVALID;
    az_select_args a;
    a.batch = p->batch_size; a.coef = p->exploration_coef;
    a.noise_scale = p->noise_scale; a.noise_alpha = p->noise_alpha; a.root_mode = 0;
    return az_select_launch(e, a, stream);
}

int az_leaf_moves(az_engine *e, void *stream)
{
    if (!e) return AZ_E_INVALID;
    AZ_LAUNCH(k_leaf_moves, e, stream);
}

static int az_expand_launch(az_engine *e, const float *value_dev, const float *prior_dev,
                            int prior_kind, int root_mode, void *stream)
{
    if (!e || (prior_kind != AZ_PRIOR_PROBS && prior_kind != AZ_PRIOR_LOGITS)) return AZ_E_INVALID;
    az_expand_args a;
    a.batch = root_mode ? 1 : e->B;
    a.prior_kind = prior_kind;
    /* caller arrays hold the rows of the current game window only */
    a.value = value_dev ? value_dev - (size_t)e->g0 * e->B : e->value;
    a.prior = prior_dev ? prior_dev - (size_t)e->g0 * e->B * e->nn : e->prior;
    a.root_mode = root_mode;
    if (e->NW <= 4) {
        AZ_LAUNCH(k_expand_backup<4>, e, stream, a);
    } else {
        AZ_LAUNCH(k_expand_backup<12>, e, stream, a);
    }
}

int az_mcts_expand_backup(az_engine *e, const float *value_dev, const float *prior_dev,
                          int prior_kind, void *stream)
{
    return az_expand_launch(e, value_dev, prior_dev, prior_kind, 0, stream);
}

int az_mcts_expand_root(az_engine *e, const float *prior_dev, int prior_kind, void *stream)
{
    return az_expand_launch(e, NULL, prior_dev, prior_kind, 1, stream);
}

int az_root_stats(az_engine *e, float *visits_dev, float *total_value_dev, float *prior_dev,
                  int32_t *num_children_dev, float *root_nw_dev, int64_t *num_nodes_dev,
                  void *stream)
{
    if (!e) return AZ_E_INVALID;
    AZ_LAUNCH(k_root_stats, e, stream, visits_dev, total_value_dev, prior_dev, num_children_dev,
              root_nw_dev, num_nodes_dev);
}

int az_engine_set_window(az_engine *e, int first_game, int num_games)
{
    if (!e) return AZ_E_INVALID;
    if (num_games <= 0) { first_game = 0; num_games = e->G; }
    if (first_game < 0 || first_game + num_games > e->G) return AZ_E_INVALID;
    e->g0 = first_game;
    e->g1 = first_game + num_games;
    return AZ_OK;
}

int az_engine_set_reflect(az_engine *e, int on)
{
    if (!e) return AZ_E_INVALID;
    e->reflect = on != 0;
    return AZ_OK;
}

int az_engine_set_playout_cap(az_engine *e, float full_search_prob, int fast_descents)
{
    if (!e || !(full_search_prob >= 0.0f)) return AZ_E_INVALID;     // (NaN fails the test)
    if (full_search_prob >= 1.0f) {
        e->fast_descents = 0;
        e->full_thresh = 0;
        return AZ_OK;
    }
    if (fast_descents < 1) return AZ_E_INVALID;
    e->fast_descents = fast_descents;
    // coin < p * 2^32 for an integer coin is coin < ceil(p * 2^32); exact in double
    e->full_thresh = (unsigned long long)ceil((double)full_search_prob * 4294967296.0);
    return AZ_OK;
}

int az_engine_set_resign(az_engine *e, float threshold, float disable_prob)
{
    // (NaN fails every test)
    if (!e || !(threshold <= 1.0f) || !(disable_prob >= 0.0f && disable_prob <= 1.0f))
        return AZ_E_INVALID;
    e->resign_on = threshold > -1.0f;
    e->resign_thresh = e->resign_on ? threshold : 0.0f;
    // coin < p * 2^32 for an integer coin is coin < ceil(p * 2^32); exact in double
    e->calib_thresh = e->resign_on ? (unsigned long long)ceil((double)disable_prob * 4294967296.0) : 0ull;
    return AZ_OK;
}

int az_engine_set_forced_playouts(az_engine *e, float k, float exploration_coef)
{
    if (!e || !(k >= 0.0f) || !isfinite(k) || !(exploration_coef >= 0.0f) || !isfinite(exploration_coef))
        return AZ_E_INVALID;
    e->forced_k = k;
    e->prune_coef = k != 0.0f ? exploration_coef : 0.0f;
    return AZ_OK;
}

int az_mcts_root_uniform(az_engine *e, void *stream)
{
    if (!e) return AZ_E_INVALID;
    AZ_LAUNCH(k_root_uniform, e, stream);
}

int az_tree_move(az_engine *e, const int32_t *move_ids_dev, void *stream)
{
    if (!e || !move_ids_dev) return AZ_E_INVALID;
    AZ_LAUNCH(k_tree_move, e, stream, move_ids_dev);
}

int az_status(az_engine *e, int32_t *status_dev, void *stream)
{
    if (!e || !status_dev) return AZ_E_INVALID;
    az_device_guard guard(e->device);
    k_status<<<(e->G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*e, status_dev);
    return az_check(cudaGetLastError());
}

int az_stub_eval(az_engine *e, int mode, void *stream)
{
    if (!e || mode < 0 || mode > 2) return AZ_E_INVALID;
    AZ_LAUNCH(k_stub_eval, e, stream, mode);
}

int az_noise_sample(az_engine *e, float alpha, int k, int sim, float *out_dev, void *stream)
{
    if (!e || !out_dev || k < 1 || k > e->nn || alpha <= 0.0f) return AZ_E_INVALID;
    AZ_LAUNCH(k_noise_sample, e, stream, alpha, k, sim, out_dev);
}

int az_replay_collate(const uint8_t *rows_dev, int row_bytes, const int64_t *index_dev, int count,
                      int board_size, int32_t *board_dev, int32_t *moves_dev, float *probs_dev,
                      float *reward_dev, int64_t *color_dev, int64_t *result_dev,
                      int32_t *num_moves_dev, void *stream)
{
    if (!rows_dev || !index_dev || !board_dev || !moves_dev || !probs_dev || !reward_dev ||
        !color_dev || !result_dev || !num_moves_dev || board_size < 2 || board_size > 19 || count < 0)
        return AZ_E_INVALID;
    const int nn = board_size * board_size, cs = (nn + 15) & ~15;
    if (row_bytes < (int)sizeof(az_row_header) + cs + 4 * nn) return AZ_E_INVALID;
    if (count == 0) return AZ_OK;
    k_replay_collate<<<(count + AZ_WARPS_PER_CTA - 1) / AZ_WARPS_PER_CTA, AZ_WARPS_PER_CTA * 32, 0,
                       (cudaStream_t)stream>>>(rows_dev, row_bytes, index_dev, count, board_size, cs,
                                               board_dev, moves_dev, probs_dev, reward_dev, color_dev,
                                               result_dev, num_moves_dev);
    return az_check(cudaGetLastError());
}

int az_batch_reflect(int32_t *board_dev, int32_t *moves_dev, float *probs_dev,
                     const uint8_t *coins_dev, int count, int board_size, int width, int ld,
                     void *stream)
{
    if (!board_dev || !moves_dev || !probs_dev || !coins_dev || board_size < 2 || board_size > 19 ||
        count < 0 || width < 0 || width > board_size * board_size || ld < width)
        return AZ_E_INVALID;
    if (count == 0) return AZ_OK;
    k_batch_reflect<<<(count + AZ_WARPS_PER_CTA - 1) / AZ_WARPS_PER_CTA, AZ_WARPS_PER_CTA * 32, 0,
                      (cudaStream_t)stream>>>(board_dev, moves_dev, probs_dev, coins_dev, count,
                                              board_size * board_size, width, ld);
    return az_check(cudaGetLastError());
}

int az_nn_stem(const int8_t *cells_dev, int cell_stride, int board_size, int64_t num_boards,
               const void *table_dev, const float *bias_dev, void *out_dev, int channels,
               int padded_layout, void *stream)
{
    return az_nn_stem_live(cells_dev, cell_stride, board_size, num_boards, table_dev, bias_dev, out_dev,
                           channels, padded_layout, nullptr, stream);
}

int az_nn_stem_live(const int8_t *cells_dev, int cell_stride, int board_size, int64_t num_boards,
                    const void *table_dev, const float *bias_dev, void *out_dev, int channels,
                    int padded_layout, const int32_t *live_rows_dev, void *stream)
{
    if (live_rows_dev && !padded_layout) return AZ_E_UNSUPPORTED;
    if (padded_layout && channels != 64) return AZ_E_UNSUPPORTED;
    if (!cells_dev || !table_dev || !bias_dev || !out_dev || board_size < 2 || board_size > 19 ||
        channels < 8 || channels > AZ_NN_MAXC || (channels & 7) || num_boards < 0 ||
        cell_stride < board_size * board_size)
        return AZ_E_INVALID;
    if (num_boards == 0) return AZ_OK;
    if (padded_layout) {
        const int bpg = 128 / (board_size + 1);
        const size_t smem = AZ_STEM_SLAB_SMEM(board_size, bpg);
        static bool attr_set[AZ_MAX_DEVICES];       // the opt-in is per device
        const int dev = az_current_device();
        if (!attr_set[dev]) {
            int rc = az_check(cudaFuncSetAttribute(k_nn_stem_slab, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   AZ_STEM_SLAB_SMEM(19, 6)));
            if (rc != AZ_OK) return rc;
            attr_set[dev] = true;
        }
        long long blocks = (num_boards + bpg - 1) / bpg;
        if (blocks > az_sm_count(dev) * 6) blocks = az_sm_count(dev) * 6;
        k_nn_stem_slab<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(
            cells_dev, cell_stride, board_size, (long long)num_boards, (const uint16_t *)table_dev,
            bias_dev, (uint16_t *)out_dev, live_rows_dev);
        return az_check(cudaGetLastError());
    }
    const int pnn = (board_size + 2) * (board_size + 2);
    const int nn = board_size * board_size;
    const size_t smem = (size_t)36 * channels * 2 + (size_t)((nn + 1) & ~1) * 2 +
                        (size_t)AZ_NN_STEM_BOARDS * pnn;
    if (256 % (channels >> 3)) return AZ_E_UNSUPPORTED;
    long long blocks = (num_boards + AZ_NN_STEM_BOARDS - 1) / AZ_NN_STEM_BOARDS;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_nn_stem<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(
        cells_dev, cell_stride, board_size, (long long)num_boards, (const uint16_t *)table_dev,
        bias_dev, (uint16_t *)out_dev, channels, padded_layout);
    return az_check(cudaGetLastError());
}

int az_nn_heads(const void *x_dev, int64_t positions, const float *w_dev, const float *b_dev,
                void *out_dev, int64_t out_board_stride, int channels, int heads, int padded_board_size,
                void *stream)
{
    return az_nn_heads_live(x_dev, positions, w_dev, b_dev, out_dev, out_board_stride, channels, heads,
                            padded_board_size, nullptr, stream);
}

int az_nn_heads_live(const void *x_dev, int64_t positions, const float *w_dev, const float *b_dev,
                     void *out_dev, int64_t out_board_stride, int channels, int heads, int padded_board_size,
                     const int32_t *live_rows_dev, void *stream)
{
    if (live_rows_dev && !padded_board_size) return AZ_E_UNSUPPORTED;
    if (out_board_stride && !padded_board_size) return AZ_E_UNSUPPORTED;
    if (padded_board_size && channels != 64) return AZ_E_UNSUPPORTED;
    if (!x_dev || !w_dev || !b_dev || !out_dev || channels < 8 || channels > AZ_NN_MAXC ||
        (channels & 7) || positions < 0)
        return AZ_E_INVALID;
    if (heads != 6) return AZ_E_UNSUPPORTED;   /* value_chans 2 + policy_chans 4, network.py:123 */
    if (((channels >> 3) & ((channels >> 3) - 1)) || (channels >> 3) < 4)
        return AZ_E_UNSUPPORTED;               /* lanes per position: power of two, >= heads/2 */
    if (positions == 0) return AZ_OK;
    if (padded_board_size) {
        const int n = padded_board_size, bpg = 128 / (n + 1);
        if (n < 2 || n > 19 || positions % (n * n)) return AZ_E_INVALID;
        if (out_board_stride == 0) out_board_stride = (int64_t)n * n * heads;
        if (out_board_stride < n * n * heads || (out_board_stride & 1)) return AZ_E_INVALID;
        const long long boards = positions / (n * n);
        long long blocks = (boards + bpg - 1) / bpg * n;
        if (blocks > 148 * 8) blocks = 148 * 8;
        k_nn_heads_slab<6><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            (const uint16_t *)x_dev, boards, n, w_dev, b_dev, (uint16_t *)out_dev, (long long)out_board_stride,
            live_rows_dev);
        return az_check(cudaGetLastError());
    }
    long long blocks = (positions * (channels >> 3) + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_nn_heads<6><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const uint16_t *)x_dev, (long long)positions, w_dev, b_dev, (uint16_t *)out_dev, channels,
        padded_board_size);
    return az_check(cudaGetLastError());
}

int az_nn_tail(const void *y_dev, int64_t num_boards, int ld, int nfc2, int board_size,
               const float *fc_bias_dev, const float *w3_dev, const float *b3_dev,
               float *value_dev, int64_t value_stride, float *logits_dev, int64_t logits_stride,
               void *stream)
{
    return az_nn_tail_live(y_dev, num_boards, ld, nfc2, board_size, fc_bias_dev, w3_dev, b3_dev, value_dev,
                           value_stride, logits_dev, logits_stride, nullptr, stream);
}

int az_nn_tail_live(const void *y_dev, int64_t num_boards, int ld, int nfc2, int board_size,
                    const float *fc_bias_dev, const float *w3_dev, const float *b3_dev,
                    float *value_dev, int64_t value_stride, float *logits_dev, int64_t logits_stride,
                    const int32_t *live_rows_dev, void *stream)
{
    const int nn = board_size * board_size;
    if (!y_dev || !fc_bias_dev || !w3_dev || !b3_dev || board_size < 2 || board_size > 19 ||
        num_boards < 0 || nfc2 < 2 || (nfc2 & 1) || ld < nfc2 + nn || (ld & 1) ||
        (logits_dev && logits_stride < nn) || (value_dev && value_stride < 1))
        return AZ_E_INVALID;
    if (num_boards == 0) return AZ_OK;
    long long blocks = (num_boards + 7) / 8;
    const int cap = az_sm_count(az_current_device()) * 16;
    if (blocks > cap) blocks = cap;
    k_nn_tail<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const uint16_t *)y_dev, (long long)num_boards, ld, nfc2, nn, fc_bias_dev, w3_dev, b3_dev,
        value_dev, (long long)value_stride, logits_dev, (long long)logits_stride, live_rows_dev);
    return az_check(cudaGetLastError());
}

int az_nn_tower_group(int board_size)
{
    /* boards that share one 128-row slab */
    return (board_size < 2 || board_size > 19) ? AZ_E_INVALID : 128 / (board_size + 1);
}

int az_nn_tower_halo(int board_size)
{
    return (board_size < 2 || board_size > 19) ? AZ_E_INVALID : AZT_HALO;
}

int64_t az_nn_tower_rows(int board_size, int64_t num_boards)
{
    if (board_size < 2 || board_size > 19 || num_boards < 0) return AZ_E_INVALID;
    const int bpg = 128 / (board_size + 1);
    const int64_t groups = (num_boards + bpg - 1) / bpg;
    /* 8 zero rows, n slabs of 128 rows per group, 16 zero rows */
    return AZT_HALO + groups * board_size * 128 + 16;
}

static int azt_launch(azt_params &p, bool resid, void *stream)
{
    static int debug = -1;                  /* probe switches (az_tower.cuh), read once */
    if (debug < 0) { const char *dbg = getenv("AZT_DEBUG"); debug = dbg ? atoi(dbg) : 0; }
    p.debug = debug;
    static bool attr_set[AZ_MAX_DEVICES];           // the shared-memory opt-in is per device
    const int dev = az_current_device();
    const int sm_count = az_sm_count(dev);
    if (!attr_set[dev]) {
        int rc = az_check(cudaFuncSetAttribute(k_conv3x3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AZT_SMEM_BYTES));
        if (rc == AZ_OK)
            rc = az_check(cudaFuncSetAttribute(k_conv3x3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, AZT_SMEM_BYTES));
        if (rc != AZ_OK) return rc;
        attr_set[dev] = true;
    }
    const unsigned grid = (unsigned)(p.groups < sm_count ? p.groups : sm_count);
    if (resid)
        k_conv3x3<true><<<grid, AZT_THREADS, AZT_SMEM_BYTES, (cudaStream_t)stream>>>(p);
    else
        k_conv3x3<false><<<grid, AZT_THREADS, AZT_SMEM_BYTES, (cudaStream_t)stream>>>(p);
    return az_check(cudaGetLastError());
}

int az_nn_conv3x3(const void *x_dev, const void *w_dev, const float *bias_dev, const void *resid_dev,
                  void *out_dev, int board_size, int64_t num_boards, void *stream)
{
    if (!x_dev || !w_dev || !bias_dev || !out_dev || board_size < 2 || board_size > 19 || num_boards < 0)
        return AZ_E_INVALID;
    if (num_boards == 0) return AZ_OK;
    azt_params p = {};
    p.x = (const uint8_t *)x_dev; p.w = (const uint8_t *)w_dev; p.bias = bias_dev;
    p.resid = (const uint8_t *)resid_dev; p.out = (uint8_t *)out_dev;
    p.n = board_size; p.bpg = 128 / (board_size + 1);
    p.groups = (num_boards + p.bpg - 1) / p.bpg;
    return azt_launch(p, resid_dev != nullptr, stream);
}

static int azb_max_clusters[AZ_MAX_DEVICES];

int az_nn_resblock_clusters(void)
{
    /* diagnostic: clusters of two CTAs az_nn_resblock found resident at once on the current
     * device (0 before its first launch there) */
    return azb_max_clusters[az_current_device()];
}

size_t az_nn_resblock_scratch_bytes(void)
{
    /* the intermediate slabs travel through distributed shared memory, never global memory */
    return 0;
}

static int azb_launch(void *x_dev, const void *w_dev, const float *bias_dev, int board_size,
                      int64_t num_boards, int passes, const int32_t *live_rows_dev, void *stream)
{
    azb_params p = {};
    p.live = live_rows_dev;
    p.x = (uint8_t *)x_dev; p.w = (const uint8_t *)w_dev; p.bias = bias_dev;
    p.n = board_size; p.bpg = 128 / (board_size + 1);
    p.groups = (num_boards + p.bpg - 1) / p.bpg;
    p.passes = passes;
    // clusters of two CTAs (one per SM) that can be resident at once on this device
    int *max_clusters = azb_max_clusters;
    const int dev = az_current_device();
    if (max_clusters[dev] == 0) {
        int rc = az_check(cudaFuncSetAttribute(k_resblock, cudaFuncAttributeMaxDynamicSharedMemorySize, AZB_SMEM_BYTES));
        if (rc != AZ_OK) return rc;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * (unsigned)(az_sm_count(dev) / 2));
        cfg.blockDim = dim3(AZB_THREADS);
        cfg.dynamicSmemBytes = AZB_SMEM_BYTES;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        int nc = 0;
        rc = az_check(cudaOccupancyMaxActiveClusters(&nc, k_resblock, &cfg));
        if (rc != AZ_OK) return rc;
        if (nc < 1) return AZ_E_UNSUPPORTED;
        if (nc > az_sm_count(dev) / 2) nc = az_sm_count(dev) / 2;
        max_clusters[dev] = nc;
    }
    const long long clusters = p.groups < max_clusters[dev] ? p.groups : max_clusters[dev];
    k_resblock<<<(unsigned)(2 * clusters), AZB_THREADS, AZB_SMEM_BYTES, (cudaStream_t)stream>>>(p);
    return az_check(cudaGetLastError());
}

int az_nn_resblock(void *x_dev, const void *w_dev, const float *bias_dev, void *scratch_dev,
                   int board_size, int64_t num_boards, void *stream)
{
    return az_nn_resblocks(x_dev, w_dev, bias_dev, scratch_dev, board_size, num_boards, 1, stream);
}

int az_nn_resblocks(void *x_dev, const void *w_dev, const float *bias_dev, void *scratch_dev,
                    int board_size, int64_t num_boards, int num_blocks, void *stream)
{
    return az_nn_resblocks_live(x_dev, w_dev, bias_dev, scratch_dev, board_size, num_boards, num_blocks,
                                nullptr, stream);
}

int az_nn_resblocks_live(void *x_dev, const void *w_dev, const float *bias_dev, void *scratch_dev,
                         int board_size, int64_t num_boards, int num_blocks, const int32_t *live_rows_dev,
                         void *stream)
{
    if (!x_dev || !w_dev || !bias_dev || board_size < 2 || board_size > 19 || num_boards < 0 || num_blocks < 0)
        return AZ_E_INVALID;
    if (num_boards == 0) return AZ_OK;
    for (int b = 0; b < num_blocks; b += AZB_MAXPASS) {
        const int passes = num_blocks - b < AZB_MAXPASS ? num_blocks - b : AZB_MAXPASS;
        int rc = azb_launch(x_dev, (const uint8_t *)w_dev + (size_t)b * 2 * AZT_WBYTES, bias_dev + (size_t)b * 2 * AZT_C,
                            board_size, num_boards, passes, live_rows_dev, stream);
        if (rc != AZ_OK) return rc;
    }
    return AZ_OK;
}

static_assert(AZB_SMEM_BYTES + 4096 <= 232448, "k_resblock: dynamic + static shared memory per CTA");

int az_play_commit(az_engine *e, const az_play_params *p, int32_t *chosen_dev, void *stream)
{
    if (!e || !p) return AZ_E_INVALID;
    if (p->collect_replay && e->hist_rows == 0) return AZ_E_INVALID;
    AZ_LAUNCH(k_play_commit, e, stream, *p, chosen_dev);
}

int az_replay_clear(az_engine *e, void *stream)
{
    if (!e) return AZ_E_INVALID;
    az_device_guard guard(e->device);
    k_replay_clear<<<1, 32, 0, (cudaStream_t)stream>>>(*e);
    return az_check(cudaGetLastError());
}

} // extern "C"
