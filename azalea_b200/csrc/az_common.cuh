// az_common.cuh -- engine layout + warp-level device helpers (sm_100a).
//
// One warp owns one game.  Boards are bit-packed and *lane-distributed*:
// lane w holds 32-tile word w of the X mask and of the O mask (11x11 -> 4
// words, 19x19 -> 12 words), so setting a stone is a predicated OR on one
// lane, the k-th empty tile is a popc + short shuffle scan + ballot, and the
// winner test re-slices the mover's mask into one row per lane and floods it
// with two shuffles per step.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/azalea_b200.h"

#define AZ_FULL 0xffffffffu
#define AZ_UNEVAL 0xffffffffu       // link of an unevaluated node (search_tree.py:263 num_children = -1)
#define AZ_LINK_KBITS 9             // link = first_child << 9 | num_children
#define AZ_LINK_KMASK 511u
#define AZ_MAX_NODE ((1 << 23) - 1) // node ids are 23 bits (path entry = node | tile << 23)
#define AZ_WARPS_PER_CTA 4
#define AZ_META_INTS 16
#define AZ_CNT_PER_GAME 16

// meta[g][*]
enum {
    M_HALF = 0,     // which half of the ping-pong pool holds the tree
    M_TAIL = 1,     // nodes used in that half (root is node 0)
    M_COLOR = 2,    // colour to move 1/2 (hex.py:148)
    M_WINNER = 3,   // 0/1/2 (hex.py:149)
    M_PLY = 4,
    M_STATUS = 5,   // AZ_ST_*
    M_VREF_LO = 6,  // the reference's tree.num_nodes (never shrinks on re-root)
    M_VREF_HI = 7,
    M_SIM = 8,      // descents so far in this slot (noise stream counter)
    M_SERIAL = 9,   // games finished in this slot
    M_GID_LO = 10,  // global game id (Philox stream)
    M_GID_HI = 11,
    M_DRAW = 12,    // game hit max_plies without a winner (play_game.py:59-61)
    M_LAST = 13     // last tile played (-1 none)
};

struct az_engine {
    az_config cfg;
    int device;
    int G, n, nn, NW, B, C;
    int g0, g1;             // game window [g0, g1) the per-game kernels cover (az_engine_set_window)
    int reflect;            // 1: network rows in a random orientation (az_engine_set_reflect)
    int cell_stride;        // bytes per leaf board row (nn rounded up to 16)
    int path_stride;        // uint32 per descent path
    int row_bytes;          // replay row
    int hist_rows;          // rows of per-game history (max plies)
    uint32_t div_magic;     // (v * div_magic) >> 16 == v / n for v < 2048
    // device views inside the caller's block
    uint4 *nodes;           // [G][2][C] {N f32, W f32, P f32, link u32}
    uint32_t *board;        // [G][2][NW] X words, O words
    int32_t *meta;          // [G][16]
    uint32_t *path;         // [G][B][path_stride]
    int4 *leaf_info;        // [G][B]
    uint32_t *leaf_masks;   // [G][B][2][NW]
    int8_t *leaf_board;     // [G][B][cell_stride]
    int32_t *leaf_moves;    // [G][B][nn]
    float *value;           // [G][B]
    float *prior;           // [G][B][nn]
    unsigned long long *counters;   // [G][16]
    unsigned long long *globals;    // [16] (replay append cursor etc.)
    int32_t *leaf_rows;     // [G]: [g0] = live packed leaf rows of the window starting at g0
    uint8_t *hist;          // [G][hist_rows][row_bytes]
    uint8_t *replay;        // [replay_rows][row_bytes]
    az_buffer_desc desc[AZ_BUF__COUNT];
    size_t total_bytes;
};

// replay row header (48 bytes), then int8 board[cell_stride] (absolute
// view), then f32 visits[nn] by move ordinal
struct az_row_header {
    int64_t game_id;
    int32_t ply;
    int32_t color;      // GameState.color 0/1 (hex.py:57)
    int32_t num_moves;
    float reward;       // play_game.py:63-67
    int32_t result;
    float temperature;  // policy.py:142-149
    int32_t move;       // 1-based tile that was played
    int32_t move_id;    // its ordinal among the legal moves
    int32_t game_len;   // plies in the finished game
    int32_t reserved;
};

#ifdef __CUDACC__

__device__ __forceinline__ int az_lane() { return threadIdx.x & 31; }

__device__ __forceinline__ uint32_t az_fmix32(uint32_t h)
{
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}

// tiles of word `lane` that exist on an nn-tile board
__device__ __forceinline__ uint32_t az_valid_word(int lane, int nn)
{
    int lo = lane * 32;
    if (lo >= nn) return 0u;
    int c = nn - lo;
    return c >= 32 ? 0xffffffffu : ((1u << c) - 1u);
}

// index of the r-th (0-based) set bit of m; r < popc(m)
__device__ __forceinline__ int az_nth_set_bit(uint32_t m, int r)
{
    int pos = 0, t;
    t = __popc(m & 0xffffu); if (r >= t) { r -= t; pos += 16; m >>= 16; }
    t = __popc(m & 0xffu);   if (r >= t) { r -= t; pos += 8;  m >>= 8; }
    t = __popc(m & 0xfu);    if (r >= t) { r -= t; pos += 4;  m >>= 4; }
    t = __popc(m & 0x3u);    if (r >= t) { r -= t; pos += 2;  m >>= 2; }
    t = (int)(m & 1u);       if (r >= t) { pos += 1; }
    return pos;
}

// j-th empty tile in ascending order == legal_moves[j] - 1 (hex.py:151-159).
// `empty` is this lane's word of empty tiles (0 on lanes >= NW).
__device__ __forceinline__ int az_kth_empty(uint32_t empty, int j, int NW)
{
    const int lane = az_lane();
    int c = __popc(empty), incl = c;
    for (int off = 1; off < NW; off <<= 1) {
        int t = __shfl_up_sync(AZ_FULL, incl, off);
        if (lane >= off) incl += t;
    }
    uint32_t ball = __ballot_sync(AZ_FULL, incl > j);
    int src = __ffs(ball) - 1;
    int bit = az_nth_set_bit(empty, j - (incl - c));
    return __shfl_sync(AZ_FULL, lane * 32 + bit, src & 31);
}

__device__ __forceinline__ int az_count_bits(uint32_t word)
{
    return __reduce_add_sync(AZ_FULL, __popc(word));
}

// check_win, hex.py:204-231: does the component of `tile` in the mover's
// stones span rows 0..n-1 (colour 1) or columns 0..n-1 (colour 2)?
// `w` = this lane's word of the mover's mask (stone at `tile` included).
__device__ __forceinline__ bool az_hex_wins(uint32_t w, int n, uint32_t magic,
                                            int tile, int color)
{
    const int lane = az_lane();
    const uint32_t full = (1u << n) - 1u;
    // re-slice: lane r <- row r (n bits starting at bit r*n of the flat mask)
    int bitpos = lane * n, idx = bitpos >> 5;
    uint32_t lo = __shfl_sync(AZ_FULL, w, idx & 31);
    uint32_t hi = __shfl_sync(AZ_FULL, w, (idx + 1) & 31);
    uint32_t own = lane < n ? (__funnelshift_r(lo, hi, bitpos & 31) & full) : 0u;
    // cheap necessary condition: a stone in every row (X) / column (O)
    if (color == 1) {
        if ((__ballot_sync(AZ_FULL, own != 0u) & full) != full) return false;
    } else {
        if (__reduce_or_sync(AZ_FULL, own) != full) return false;
    }
    int tr = (int)(((uint32_t)tile * magic) >> 16), tc = tile - tr * n;
    uint32_t f = lane == tr ? (1u << tc) : 0u;
    for (;;) {
        // neighbours (hex.py:188-193): same row c-1,c+1; row above c,c+1;
        // row below c-1,c
        f |= own & ((f << 1) | (f >> 1));
        f |= own & ((f << 1) | (f >> 1));
        uint32_t up = __shfl_up_sync(AZ_FULL, f, 1);
        uint32_t dn = __shfl_down_sync(AZ_FULL, f, 1);
        if (lane == 0) up = 0u;
        if (lane == 31) dn = 0u;
        uint32_t nf = f | (own & ((f << 1) | (f >> 1) | up | (up >> 1) | dn | (dn << 1)));
        bool changed = __any_sync(AZ_FULL, nf != f);
        f = nf;
        if (!changed) break;
    }
    if (color == 1) {
        uint32_t rows = __ballot_sync(AZ_FULL, f != 0u);
        return (rows & 1u) && ((rows >> (n - 1)) & 1u);
    }
    uint32_t cols = __reduce_or_sync(AZ_FULL, f);
    return (cols & 1u) && ((cols >> (n - 1)) & 1u);
}

// tile (r,c) -> (n-1-c, n-1-r): HexGame.flip_player_board_moves, hex.py:105-117
__device__ __forceinline__ int az_flip_tile(int t, int n, uint32_t magic)
{
    int r = (int)(((uint32_t)t * magic) >> 16), c = t - r * n;
    return (n - 1 - c) * n + (n - 1 - r);
}

// Philox counter domains of the orientation coins (word w; the root noise uses 0xD1C10000)
#define AZ_REFLECT_DOMAIN 0x5EF1EC70u
#define AZ_REFLECT_ROOT_DOMAIN 0x5EF1EC71u
#define AZ_LEAF_REFLECTED (1 << AZ_LEAF_REFLECTED_BIT)

// Hex's one rule-preserving symmetry, the 180-degree rotation (i, j) -> (n-1-i, n-1-j)
__device__ __forceinline__ int az_rot_tile(int t, int nn) { return nn - 1 - t; }

__device__ __forceinline__ uint32_t az_orderable(float x)
{
    uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ uint4 az_philox(uint4 c, uint2 k)
{
#pragma unroll
    for (int i = 0; i < 10; i++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}

// 7 rounds: the fewest that still pass BigCrush (Salmon et al., SC'11);
// used for the per-simulation root noise, where the generator is the cost
__device__ __forceinline__ uint4 az_philox7(uint4 c, uint2 k)
{
#pragma unroll
    for (int i = 0; i < 7; i++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float az_u01(uint32_t r)     // (0,1)
{
    return ((float)(r >> 8) + 0.5f) * (1.0f / 16777216.0f);
}

#endif // __CUDACC__
