// az_nn_glue.cuh -- the evaluator's input and output glue (sm_100a).
//
// The 6x64 tower itself stays a library call (cuDNN, by design); these are
// the two ends of it that the library runs badly (profiles/r01_nn_launches):
//
//  k_nn_stem   network.py:138-142 + :71  Embedding(3,4) -> conv3x3(4->C) -> BN
//              -> ReLU.  A cell has 3 possible values, so the whole thing is a
//              table: out[p][c] = relu(bias[c] + sum_tap T[tap][cell(p+tap)][c])
//              with T = conv weights x embedding, BN folded.  Reads the int8
//              boards k_select wrote, writes bf16 NHWC activations.  HBM-bound:
//              n*n*C*2 bytes written per board (cuDNN: 0.81 ms, a K=36 GEMM
//              through a legacy kernel plus a channel-padding pass).
//  k_nn_heads  network.py:75-76,82-83  both 1x1 head convolutions (C -> 2 + 4)
//              + BN + ReLU in one pass over the tower output.  HBM-bound:
//              n*n*C*2 bytes read per board (library: 0.53 ms for an N=6 GEMM).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define AZ_NN_MAXC 128
#define AZ_NN_STEM_BOARDS 4

__device__ __forceinline__ void az_bf16x8_to_f32(const uint4 &v, float (&f)[8])
{
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        f[2 * i] = __uint_as_float(w[i] << 16);
        f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

__device__ __forceinline__ uint32_t az_pack_bf16x2(float lo, float hi)
{
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&p);
}

__device__ __forceinline__ long long az_min_ll(long long a, long long b) { return a < b ? a : b; }

// table: bf16 [9][4][C] (tap-major; value 3 = off board = zeros), bias f32 [C].
// Thread = (position lane, channel group of 8): 256 threads = (256 / groups)
// positions x groups.  Table and a per-position offset list live in shared
// memory, so the inner loop is 9 x (1 byte LDS + 16 B LDS + unpack + 8 FADD).
__global__ void __launch_bounds__(256)
k_nn_stem(const int8_t *__restrict__ cells, int cell_stride, int n, long long N,
          const uint16_t *__restrict__ table, const float *__restrict__ bias,
          uint16_t *__restrict__ out, int C, int padded)
{
    // padded != 0: write the tower's slab layout (az_tower.cuh): row 8 +
    // 128 * ((b / bpg) * (n+1) + y) + (b % bpg) * (n+1) + x, bpg = 128 / (n+1),
    // 16-byte chunk j at chunk j ^ (row & 7); C must be 64
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t *stab = reinterpret_cast<uint16_t *>(smem_raw);                 // 36*C bf16
    uint16_t *spos = reinterpret_cast<uint16_t *>(smem_raw + 36 * C * 2);     // nn offsets (padded to even)
    const int nn = n * n, pn = n + 2, pnn = pn * pn, pn1 = n + 1;
    int8_t *scell = reinterpret_cast<int8_t *>(smem_raw + 36 * C * 2 + ((nn + 1) & ~1) * 2);
    const int groups = C >> 3;
    const int cg = threadIdx.x % groups, tp = threadIdx.x / groups, ppt = blockDim.x / groups;
    for (int i = threadIdx.x; i < 36 * C; i += blockDim.x) stab[i] = table[i];
    for (int i = threadIdx.x; i < nn; i += blockDim.x)
        spos[i] = (uint16_t)((i / n) * pn + (i % n));       // top-left neighbour in the padded board
    float b8[8];
#pragma unroll
    for (int k = 0; k < 8; k++) b8[k] = bias[cg * 8 + k];
    const uint16_t *trow = stab + cg * 8;
    for (long long b0 = (long long)blockIdx.x * AZ_NN_STEM_BOARDS; b0 < N;
         b0 += (long long)gridDim.x * AZ_NN_STEM_BOARDS) {
        __syncthreads();
        // stage the boards with a border of "off board" cells
        for (int i = threadIdx.x; i < AZ_NN_STEM_BOARDS * pnn; i += blockDim.x) {
            const int q = i / pnn, r = (i % pnn) / pn - 1, c = (i % pnn) % pn - 1;
            int8_t v = 3;
            if (b0 + q < N && r >= 0 && r < n && c >= 0 && c < n)
                v = cells[(b0 + q) * cell_stride + r * n + c];
            scell[i] = v;
        }
        __syncthreads();
#pragma unroll 1
        for (int q = 0; q < AZ_NN_STEM_BOARDS; q++) {
            if (b0 + q >= N) break;
            uint16_t *orow = out + (b0 + q) * (long long)nn * C + cg * 8;
            const int bpg = 128 / pn1;
            const long long prow0 = 8 + ((b0 + q) / bpg) * (long long)n * 128 + ((b0 + q) % bpg) * pn1;
            for (int p = tp; p < nn; p += ppt) {
                const int8_t *sc = scell + q * pnn + spos[p];
                float acc[8];
#pragma unroll
                for (int k = 0; k < 8; k++) acc[k] = b8[k];
#pragma unroll
                for (int tap = 0; tap < 9; tap++) {
                    const int v = sc[(tap / 3) * pn + (tap % 3)];
                    const uint4 t = *reinterpret_cast<const uint4 *>(trow + (tap * 4 + v) * C);
                    float f[8];
                    az_bf16x8_to_f32(t, f);
#pragma unroll
                    for (int k = 0; k < 8; k++) acc[k] += f[k];
                }
                uint4 o;
                o.x = az_pack_bf16x2(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f));
                o.y = az_pack_bf16x2(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f));
                o.z = az_pack_bf16x2(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f));
                o.w = az_pack_bf16x2(fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f));
                if (padded) {
                    // spos[p] = y * (n+2) + x  ->  y * 128 + x
                    const long long R = prow0 + (spos[p] / pn) * 128 + spos[p] % pn;
                    *reinterpret_cast<uint4 *>(out + R * 64 + ((cg ^ (int)(R & 7)) << 3)) = o;
                } else {
                    *reinterpret_cast<uint4 *>(orow + (long long)p * C) = o;
                }
            }
        }
    }
}

// x: bf16 [P][C] (NHWC positions), w: f32 [H][C], b: f32 [H], out: bf16 [P][H].
// `groups` = C/8 lanes share a position: each lane loads one 16-byte slice
// (fully coalesced), keeps its 8 x H weights in registers, and the partial
// dot products are summed across the group by xor-shuffles.  groups must be
// a power of two <= 32 (C in {8,16,32,64,128,256}); H even.
template <int H>
__global__ void __launch_bounds__(256)
k_nn_heads(const uint16_t *__restrict__ x, long long P, const float *__restrict__ w,
           const float *__restrict__ b, uint16_t *__restrict__ out, int C, int padded_n)
{
    // padded_n != 0: x is in the tower's slab layout (az_tower.cuh) for board
    // size padded_n (C == 64); positions are still counted over real tiles
    const int groups = C >> 3;
    const int lane = threadIdx.x & 31, cg = lane % groups, sub = lane / groups;
    const int ppw = 32 / groups;                        // positions per warp per step
    float wr[H][8], br[H];
#pragma unroll
    for (int h = 0; h < H; h++) {
        br[h] = b[h];
#pragma unroll
        for (int k = 0; k < 8; k++) wr[h][k] = w[h * C + cg * 8 + k];
    }
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    constexpr int U = 4;                                // independent loads in flight per lane
    for (long long p0 = warp * ppw * U; p0 < P; p0 += nwarps * ppw * U) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long long p = p0 + u * ppw + sub;
            if (p < P && padded_n) {
                const int nn = padded_n * padded_n, pn1 = padded_n + 1;
                const long long bd = p / nn;
                const int q = (int)(p - bd * nn);
                const int bpg = 128 / pn1;
                const long long R = 8 + ((bd / bpg) * padded_n + q / padded_n) * 128 + (bd % bpg) * pn1 + q % padded_n;
                v[u] = *reinterpret_cast<const uint4 *>(x + R * 64 + ((cg ^ (int)(R & 7)) << 3));
            } else {
                v[u] = p < P ? *reinterpret_cast<const uint4 *>(x + p * C + cg * 8) : make_uint4(0, 0, 0, 0);
            }
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long long p = p0 + u * ppw + sub;
            float f[8], acc[H];
            az_bf16x8_to_f32(v[u], f);
#pragma unroll
            for (int h = 0; h < H; h++) {
                acc[h] = 0.f;
#pragma unroll
                for (int k = 0; k < 8; k++) acc[h] = fmaf(f[k], wr[h][k], acc[h]);
            }
            for (int off = 1; off < groups; off <<= 1)
#pragma unroll
                for (int h = 0; h < H; h++) acc[h] += __shfl_xor_sync(0xffffffffu, acc[h], off);
            if (p < P && cg < H / 2) {
                // lane cg of the group writes outputs 2cg, 2cg+1
                float lo = 0.f, hi = 0.f;
#pragma unroll
                for (int h = 0; h < H; h += 2)
                    if (cg == h / 2) { lo = acc[h] + br[h]; hi = acc[h + 1] + br[h + 1]; }
                reinterpret_cast<uint32_t *>(out + p * H)[cg] =
                    az_pack_bf16x2(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Slab-layout versions (the tcgen05 tower, az_tower.cuh; C == 64).  Both walk
// the activation buffer in memory order -- one block per 128-row slab -- so no
// thread ever divides a position index, and every warp access is 512
// contiguous bytes.
//
// k_nn_stem_slab: a block takes a whole board group (bpg boards, n slabs).  The
// three horizontal taps of a kernel row are one lookup: code = v(x-1) + 4 v(x)
// + 16 v(x+1) indexes T3[dy][code][c] = sum_dx T[dy*3+dx][v_dx][c] (bf16, 24 KB
// of shared memory, built once per block), and the three codes of a cell are
// one packed word, so a 16-byte output chunk is 1 LDS.32 + 3 conflict-free
// LDS.128 + 16 FADD instead of nine byte loads and nine table lookups (the bias
// rides on the centre row's entries, ReLU on the bf16 conversion).
#define AZ_STEM_SLAB_ITEMS(n, bpg) ((bpg) * ((n) + 2) * ((n) + 2))
#define AZ_STEM_SLAB_SMEM(n, bpg) \
    (3 * 64 * 64 * 2 + (bpg) * (n) * (n) * 4 + ((AZ_STEM_SLAB_ITEMS(n, bpg) + 15) & ~15) + \
     2 * ((AZ_STEM_SLAB_ITEMS(n, bpg) + 7) & ~7) + 2 * (((bpg) * (n) * (n) + 7) & ~7))

__global__ void __launch_bounds__(256)
k_nn_stem_slab(const int8_t *__restrict__ cells, int cell_stride, int n, long long N,
               const uint16_t *__restrict__ table, const float *__restrict__ bias,
               uint16_t *__restrict__ out, const int *__restrict__ live)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // packed leaves (AZ_CFG_PACK_LEAVES): only the first *live rows of this batch hold boards.
    // The groups they occupy are written whole -- rows past *live as empty boards -- so that the
    // tower never runs over activations left behind by an earlier, larger batch.
    const long long Nall = N;
    if (live != nullptr) N = az_min_ll(N, (long long)*live);
    uint16_t *t3 = reinterpret_cast<uint16_t *>(smem_raw);              // [3 dy][64 codes][64 c]
    uint32_t *scode = reinterpret_cast<uint32_t *>(smem_raw + 3 * 64 * 64 * 2);      // [bpg][n][n]
    const int pn = n + 2, pn1 = n + 1, bpg = 128 / pn1, items = bpg * pn * pn, ncell = bpg * n * n;
    int8_t *scell = reinterpret_cast<int8_t *>(scode + ncell);          // [bpg][n + 2][n + 2]
    // index arithmetic of the two staging passes, done once per block:
    // lsrc[i] = offset of padded cell i in the group's boards (0xffff: border), ltl[i] = padded
    // index of the top-left neighbour of cell i
    uint16_t *lsrc = reinterpret_cast<uint16_t *>(scell + ((items + 15) & ~15));
    uint16_t *ltl = lsrc + ((items + 7) & ~7);
    const int tid = threadIdx.x;
    for (int i = tid; i < 3 * 64 * 64; i += 256) {
        const int c = i & 63, code = (i >> 6) & 63, dy = i >> 12;
        // the centre row is always on the board: the bias rides on it
        float acc = dy == 1 ? bias[c] : 0.f;
#pragma unroll
        for (int dx = 0; dx < 3; dx++)
            acc += __uint_as_float((uint32_t)table[((dy * 3 + dx) * 4 + ((code >> (2 * dx)) & 3)) * 64 + c] << 16);
        t3[i] = __bfloat16_as_ushort(__float2bfloat16_rn(acc));
    }
    for (int i = tid; i < items; i += 256) {
        const int b = i / (pn * pn), r = (i / pn) % pn - 1, c = i % pn - 1;
        lsrc[i] = (r >= 0 && r < n && c >= 0 && c < n) ? (uint16_t)(b * cell_stride + r * n + c) : (uint16_t)0xffff;
    }
    for (int i = tid; i < ncell; i += 256) {
        const int b = i / (n * n), r = (i / n) % n, c = i % n;
        ltl[i] = (uint16_t)((b * pn + r) * pn + c);
    }
    // this thread's chunk of the rows l = (tid >> 3) + 32 i; the physical chunk tid & 7 holds
    // the logical chunk cg (swizzle: the row's low three bits are those of l)
    const int cg = (tid & 7) ^ ((tid >> 3) & 7);
    int bl[4], co[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int l = (tid >> 3) + 32 * i;
        bl[i] = l / pn1;
        const int bx = l - bl[i] * pn1;
        co[i] = bl[i] * n * n + bx;                                     // + y * n: this cell's code word
        if (bl[i] >= bpg || bx >= n) bl[i] = 1 << 30;                   // pad cell: stays zero
    }
    const long long groups = (N + bpg - 1) / bpg;
    for (long long g = blockIdx.x; g < groups; g += gridDim.x) {
        __syncthreads();
        // the group's boards with a border of "off board" cells (value 3: zero table rows)
        const int8_t *gcells = cells + g * bpg * cell_stride;
        const int limit = (int)min((long long)bpg, N - g * bpg) * cell_stride;      // boards that exist
        for (int i = tid; i < items; i += 256) {
            const int off = lsrc[i];
            scell[i] = off < limit ? gcells[off] : (int8_t)3;
        }
        __syncthreads();
        for (int i = tid; i < ncell; i += 256) {
            const int8_t *sc = scell + ltl[i];
            uint32_t word = 0;
#pragma unroll
            for (int dy = 0; dy < 3; dy++)
                word |= (uint32_t)(sc[dy * pn] + 4 * sc[dy * pn + 1] + 16 * sc[dy * pn + 2]) << (8 * dy);
            scode[i] = word;
        }
        __syncthreads();
        const int left = (int)min((long long)bpg, Nall - g * bpg);
        for (int y = 0; y < n; y++) {
            uint16_t *slab = out + (8 + (g * n + y) * 128) * 64;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (bl[i] >= left) continue;
                const uint32_t word = scode[co[i] + y * n];
                float acc[8];
#pragma unroll
                for (int dy = 0; dy < 3; dy++) {
                    const uint4 tv = *reinterpret_cast<const uint4 *>(t3 + (dy * 64 + ((word >> (8 * dy)) & 63)) * 64 + cg * 8);
                    float f[8];
                    az_bf16x8_to_f32(tv, f);
#pragma unroll
                    for (int k = 0; k < 8; k++) acc[k] = dy ? acc[k] + f[k] : f[k];
                }
                uint4 o;
                // convert + ReLU in one instruction
                asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.x) : "f"(acc[1]), "f"(acc[0]));
                asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.y) : "f"(acc[3]), "f"(acc[2]));
                asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.z) : "f"(acc[5]), "f"(acc[4]));
                asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.w) : "f"(acc[7]), "f"(acc[6]));
                reinterpret_cast<uint4 *>(slab)[tid + 256 * i] = o;
            }
        }
    }
}

// k_nn_heads_slab: the 64 -> H (<= 8) projection of a slab on mma.sync tensor cores: a warp
// takes 16 rows, four m16n8k16 steps cover the 64 channels.  No shared memory and no shuffles:
// the dot product does not care about the order of k, so thread (g = lane / 4, t = lane % 4)
// simply declares the 16 channels of the two 16-byte chunks it loads (logical chunks t and
// t + 4 of rows g and g + 8) to be its k slots, and holds the weights of the same channels
// in its B fragments.  Weights are split into bf16 hi + lo parts (two MMAs per step), so the
// result has fp32-weight accuracy like k_nn_heads.
__device__ __forceinline__ void az_mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2])
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int H>
__global__ void __launch_bounds__(256)
k_nn_heads_slab(const uint16_t *__restrict__ x, long long N, int n, const float *__restrict__ w,
                const float *__restrict__ b, uint16_t *__restrict__ out, long long ostride,
                const int *__restrict__ live)
{
    static_assert(H <= 8 && (H & 1) == 0, "heads fit one n = 8 MMA tile");
    if (live != nullptr) N = az_min_ll(N, (long long)*live);
    const int tid = threadIdx.x, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int pn1 = n + 1, bpg = 128 / pn1;
    // B fragments of column (head) g for the four k steps: step s covers channels
    // chunk * 8 + (s & 1) * 4 + {0..3} of chunk = t (s < 2) or t + 4
    uint32_t bhi[4][2], blo[4][2];
#pragma unroll
    for (int s = 0; s < 4; s++)
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const int k0 = ((s < 2 ? t : t + 4) * 8) + (s & 1) * 4 + 2 * r;
            const float w0 = g < H ? w[g * 64 + k0] : 0.f, w1 = g < H ? w[g * 64 + k0 + 1] : 0.f;
            const __nv_bfloat16 h0 = __float2bfloat16_rn(w0), h1 = __float2bfloat16_rn(w1);
            const __nv_bfloat16 l0 = __float2bfloat16_rn(w0 - __bfloat162float(h0));
            const __nv_bfloat16 l1 = __float2bfloat16_rn(w1 - __bfloat162float(h1));
            bhi[s][r] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            blo[s][r] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
        }
    const float bias0 = 2 * t < H ? b[2 * t] : 0.f, bias1 = 2 * t < H ? b[2 * t + 1] : 0.f;
    // this thread's two rows of every slab (l & 7 == g for both: same swizzle)
    int lrow[2], bl[2];
    long long off[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
        lrow[r] = (tid >> 5) * 16 + g + 8 * r;
        bl[r] = lrow[r] / pn1;
        const int bx = lrow[r] - bl[r] * pn1;
        off[r] = bl[r] * ostride + bx * H;
        if (bl[r] >= bpg || bx >= n) bl[r] = 1 << 30;                    // pad cell
        else if (2 * t >= H) bl[r] = 1 << 30;                            // columns H..7 are padding
    }
    const int c0 = t ^ g, c1 = (t + 4) ^ g;                              // physical chunks of logical t, t + 4
    const long long slabs = (N + bpg - 1) / bpg * n;
    for (long long q = blockIdx.x; q < slabs; q += gridDim.x) {
        const long long grp = q / n;
        const int y = (int)(q - grp * n);
        const uint4 *slab = reinterpret_cast<const uint4 *>(x + (8 + q * 128) * 64);
        const uint4 a00 = slab[lrow[0] * 8 + c0], a01 = slab[lrow[0] * 8 + c1];
        const uint4 a10 = slab[lrow[1] * 8 + c0], a11 = slab[lrow[1] * 8 + c1];
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        {
            const uint32_t f0[4] = {a00.x, a10.x, a00.y, a10.y}, f1[4] = {a00.z, a10.z, a00.w, a10.w};
            const uint32_t f2[4] = {a01.x, a11.x, a01.y, a11.y}, f3[4] = {a01.z, a11.z, a01.w, a11.w};
            az_mma_bf16_16816(acc, f0, bhi[0]); az_mma_bf16_16816(acc, f0, blo[0]);
            az_mma_bf16_16816(acc, f1, bhi[1]); az_mma_bf16_16816(acc, f1, blo[1]);
            az_mma_bf16_16816(acc, f2, bhi[2]); az_mma_bf16_16816(acc, f2, blo[2]);
            az_mma_bf16_16816(acc, f3, bhi[3]); az_mma_bf16_16816(acc, f3, blo[3]);
        }
        uint16_t *obase = out + grp * bpg * ostride + (long long)y * n * H;
        const long long left = N - grp * bpg;                            // boards of this group that exist
#pragma unroll
        for (int r = 0; r < 2; r++)
            if (bl[r] < left)
                reinterpret_cast<uint32_t *>(obase + off[r])[t] =
                    az_pack_bf16x2(fmaxf(acc[2 * r] + bias0, 0.f), fmaxf(acc[2 * r + 1] + bias1, 0.f));
    }
}

// ---------------------------------------------------------------------------
// k_nn_tail: everything after the merged fully connected GEMM, one warp per board.
// y bf16 [N][ld] = (head activations) x (value_fc2 | move_fc)^T WITHOUT bias:
//   columns [0, nfc2)           value_fc2 pre-activations  (network.py:78-79)
//   columns [nfc2, nfc2 + nn)   move_fc logits over tiles  (network.py:145)
// value  = tanh(value_fc3(relu(y[:nfc2] + bias)))            -> value[b * value_stride]
// logits = y[nfc2:] + bias, fp32                             -> logits[b * logits_stride + tile]
// The outputs go straight into the engine's AZ_BUF_VALUE / AZ_BUF_PRIOR rows (the
// legal-move gather and softmax happen in k_expand_backup, AZ_PRIOR_LOGITS), so no
// library elementwise kernel runs between the GEMM and the tree.
__global__ void __launch_bounds__(256)
k_nn_tail(const uint16_t *__restrict__ y, long long N, int ld, int nfc2, int nn,
          const float *__restrict__ bias, const float *__restrict__ w3, const float *__restrict__ b3,
          float *__restrict__ value, long long value_stride,
          float *__restrict__ logits, long long logits_stride, const int *__restrict__ live)
{
    if (live != nullptr) N = az_min_ll(N, (long long)*live);
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long b = warp; b < N; b += nwarps) {
        const uint32_t *row = reinterpret_cast<const uint32_t *>(y + b * ld);
        float part = 0.f;
        for (int c2 = lane; 2 * c2 < nfc2 + nn; c2 += 32) {
            const uint32_t w = row[c2];
            const float v[2] = {__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)};
#pragma unroll
            for (int h = 0; h < 2; h++) {
                // the last pair of an odd nfc2 + nn ends one column past the row: bias has
                // only nfc2 + nn elements, so it is read for real columns only
                const int c = 2 * c2 + h;
                if (c < nfc2) part = fmaf(fmaxf(v[h] + bias[c], 0.f), w3[c], part);
                else if (c < nfc2 + nn && logits) logits[b * logits_stride + (c - nfc2)] = v[h] + bias[c];
            }
        }
        for (int off = 16; off; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        if (value && lane == 0) value[b * value_stride] = tanhf(part + b3[0]);
    }
}
