// az_block.cuh -- the residual blocks of the evaluator's tower, one or all of them per launch (sm_100a):
//     x <- relu(conv2(relu(conv1(x) + b1)) + b2 + x)         (network.py:17-39, BN folded)
// on tcgen05 tensor cores, in place, reading x once and writing it once.
//
// az_tower.cuh runs a block as two launches, x -> y and y, x -> x: five passes over the
// activations per block (2 + 3), and in the power-capped steady state of the self-play step
// both launches sit on the HBM roofline (4.5 TB/s sustained, profiles/r01_*).  The
// intermediate y never needs to exist in memory.  Two things stand in the way of fusing the
// two convolutions on ONE SM: shared memory and TMEM (both layers' weights are 144 KB, and two
// accumulator rings of four blocks would split half of the N = 192 MMA windows at the ring
// end), and shared-memory BANDWIDTH: the 12 MMAs of a slab read 120 KB of operands (A 48 KB,
// the 72 KB of weights every slab) against 128 B/clock, 940 of the slab's 1152 MMA cycles --
// k_conv3x3's measured 1337 cycles per slab are exactly its 170 KB of shared-memory traffic
// per slab (operands + 18 KB input + staging tile written and read back).
//
// So the block runs on a CLUSTER OF TWO CTAs, a producer and a consumer, each with its own
// layer's weights (72 KB) and its own eight-block TMEM ring (every MMA window stays N = 192,
// cta_group::1, no split):
//
//   CTA 0 "P" (conv1):  x slabs --bulk g2s--> input ring --MMA--> TMEM --epilogue (+b1, ReLU,
//                       bf16)--> staging tile --cp.async.bulk shared::cta -> shared::cluster-->
//                       C's input ring (distributed shared memory; the copy completes, with
//                       complete_tx, on C's own mbarrier)
//   CTA 1 "C" (conv2):  --MMA--> TMEM --epilogue (+b2, + x from a bulk-loaded residual ring,
//                       ReLU)--> staging tile --bulk s2g--> x (in place).  The residual x slab
//                       is read a second time by C a few microseconds after P read it: an L2
//                       hit (126 MB L2, ~10 MB of slabs in flight on the device).
//
// HBM traffic per block is one read and one write of the activations (2 units instead of 5).
//
// Flow control between the two CTAs (mbarriers only, no cluster-scope fence on any hot path):
//   C.in_full[st]    tx barrier of stage st of C's ring; armed by C (arrive.expect_tx),
//                    completed by the bytes of P's shared-to-shared bulk copy
//   P.y_free[st]     remote arrive by C's relay once MMA2 of the slab in stage st has retired
//   P.out_empty[sb]  remote arrive by C's relay once the slab copied from P's staging tile sb
//                    has landed (the copy completes on C's barrier only, so C tells P)
// The remote arrives are RELAXED: they publish no data (the stage / tile they release was read
// by the tensor core or the copy engine, whose completion the relay has observed), and a
// release at cluster scope costs ~1000 cycles here (measured, profiles/r02_fused_block.txt).
// No tile ever mixes bulk writes with bulk reads (staging: generic writes + bulk reads;
// input rings: bulk writes + tensor-core reads).
//
// Two lessons are built in (profiles/r02_fused_block.txt has the measurements):
//  * An mbarrier arrive does NOT wait for the shared-memory loads issued before it.  The
//    residual ring's release overtook the epilogue's loads and slow warps read the slab that
//    was loaded three slabs later (~2 % of the rows wrong, nondeterministic); the release now
//    depends on the loaded registers.
//  * Anything with release semantics at cluster scope (mbarrier.arrive.release.cluster, and
//    fence.proxy.async over all state spaces) costs 1000-2000 cycles per call here, with or
//    without outstanding stores.  A variant whose P epilogue stored y straight into C's ring
//    (st.shared::cluster, fence, release arrive; C with register residuals and direct global
//    stores) was bit-exact and took 0.92 ms per block; its direct, per-row global accesses in
//    C's epilogue (32 different lines per warp instruction) alone cost 0.19 ms each way.
//
// Alternatives measured and removed (all bit-exact; where the numbers are):
//  * y from P to C through an L2-resident scratch ring in global memory (P bulk-stores the
//    staging tile, C bulk-loads it; the link carries only arrives): 8.96e6 against 9.22e6
//    simulations/s in the step (profiles/r02_fused_block.txt)
//  * y sent by P's epilogue with st.async, registers -> C's ring: 0.65 against 0.59 ms per block;
//    4 x STAS.128 per thread and slab keep P's epilogue busy 2600 cycles per slab (same file)
//  * C's epilogue reading the residual from and writing its output to global memory directly,
//    whole lines per eight lanes with an 8 x 8 shuffle transpose on each side: 0.63 against
//    0.57 ms per block, ~400 instructions per thread and slab for the transposes (same file)
//  * two storer threads per CTA (even / odd slabs): the kernel is bound elsewhere when the MMAs
//    run, and the extra warp costs 1 % (same file)
//  * the two 1x1 head convolutions fused into C's epilogue of the last pass: 3.3 % slower in the
//    step than the separate heads kernel (profiles/r02_fused_heads_ab.txt)
//
// Everything else -- slab layout, pointer-shift taps, dy stacking into a TMEM accumulator
// ring, ping-pong MMA issuers, two epilogue groups -- is az_tower.cuh's; see there.
//
// CHAINED BLOCKS (az_nn_resblocks, `passes` > 1): a board's activations depend on no other
// board, so a cluster runs block b + 1 over its own range of groups as soon as it has finished
// block b there -- no grid-wide synchronisation, and the P -> C pipeline is filled and drained
// once per launch instead of once per block (a launch costs ~14 us beyond its slabs; +4.7 %
// simulations/s in the step).  The slab index t = pass * nslabs + j simply runs on: rings,
// barrier phases and the TMEM ring continue across a pass boundary (nslabs is a multiple of the
// board size, so the board row is t % n), j addresses memory.  Added for it: all passes' biases
// in shared memory; a "weights" thread per CTA that follows every slab's MMA-retired barrier
// (a parity wait is only sound one phase away) and loads the next pass's weights when the last
// slab of a pass has retired; and s_stored, the count of output slabs whose bulk store has
// COMPLETED, kept by C's storer in both CTAs' shared memory -- P's loader (its next input) and
// C's residual loader wait for it before they read a slab again.
//
// Roles (672 threads per CTA):
//   warps 0-15   epilogue (two groups of eight on alternate output slabs)
//   warps 16,17  MMA issuers (even / odd slabs)
//   warp 18      loader: P: x chunks (144 rows); C: residual slabs (128 rows)
//   warp 19      lane 0, C: relay (slab landed -> P.out_empty; MMA2 retired -> re-arm, P.y_free)
//                lane 1, both: this CTA's weights, pass after pass
//   warp 20      storer: P: staging tile -> C's ring; C: staging tile -> x, and s_stored
#pragma once

#include "az_tower.cuh"

#define AZB_THREADS 672     // 21 warps, see Roles
#ifndef AZB_SX
#define AZB_SX 4            // P: input ring stages (x chunks, bulk loads)
#endif
#ifndef AZB_TP
#define AZB_TP 4            // P: staging tiles
#endif
#ifndef AZB_SY
#define AZB_SY 4            // C: input ring stages (y slabs copied in by P)
#endif
#ifndef AZB_SR
#define AZB_SR 2            // C: residual ring stages (x slabs, bulk loads)
#endif
#ifndef AZB_TC
#define AZB_TC 2            // C: staging tiles
#endif
#define AZB_TMAX (AZB_TP > AZB_TC ? AZB_TP : AZB_TC)
#define AZB_SMAX (AZB_SX > AZB_SY ? AZB_SX : AZB_SY)
#define AZB_SMEM_P (AZT_WBYTES + AZB_SX * AZT_CHUNK_BYTES + AZB_TP * AZT_OUT_BYTES)
#define AZB_SMEM_C (AZT_WBYTES + AZB_SY * AZT_CHUNK_BYTES + (AZB_SR + AZB_TC) * AZT_OUT_BYTES)
#define AZB_SMEM_BYTES (AZB_SMEM_P > AZB_SMEM_C ? AZB_SMEM_P : AZB_SMEM_C)
static_assert(AZB_SX <= 8 && AZB_SY <= 8, "stage reuse is tracked through the 8 MMA-retired barriers");
// Every ring that the two epilogue groups of a CTA share has an EVEN number of entries, so an
// entry always belongs to the same group (slab parity).  A parity wait then cannot be two
// phases away from its barrier: with three residual stages shared by both groups, a bulk load
// that completed late let the other group pass the wait of the NEXT use of the stage -- wrong
// residuals, and with the arrival counts mixed up, a hang or a launch failure when two
// instances ran concurrently on two streams (tools/soak.py --streams 2).
static_assert(AZB_TC % 2 == 0 && AZB_SR % 2 == 0 && AZB_TP % 2 == 0,
              "rings shared by the two epilogue groups must have an even number of entries");

#define AZB_MAXPASS 8       // residual blocks one launch can chain (their biases sit in shared memory)

struct azb_params {
    uint8_t *x;             // activations, slab layout, pre-swizzled; updated in place
    const uint8_t *w;       // [passes][2 layers][3 dx][192 = dy*64 + c_out][128 B] pre-swizzled weights
    const float *bias;      // [passes][2][64]
    int n;                  // board size
    int bpg;                // boards per group = 128 / (n+1)
    long long groups;       // board groups
    int passes;             // residual blocks to apply, one after the other (1 .. AZB_MAXPASS)
    const int *live;        // packed leaves: device count of boards that are live in this batch (or NULL: all)
};

__device__ __forceinline__ uint32_t azb_cluster_rank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

__device__ __forceinline__ void azb_cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t azb_remote(const void *p, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(azt_smem(p)), "r"(rank));
    return r;
}

// Arrive on a barrier of the other CTA without publishing anything (see the header comment).
__device__ __forceinline__ void azb_remote_arrive(uint32_t bar_cluster)
{
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}

// own shared memory -> the other CTA's shared memory; completes (complete_tx) on a barrier
// of the destination CTA
__device__ __forceinline__ void azb_bulk_s2s(uint32_t dst_cluster, const void *src, uint32_t bytes,
                                             uint32_t bar_cluster)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst_cluster), "r"(azt_smem(src)), "r"(bytes), "r"(bar_cluster) : "memory");
}

// Wait on an own barrier whose phase is completed from the other CTA (a relaxed remote arrive,
// or the bytes of its bulk copy).  The plain CTA-scope wait is enough: these barriers carry
// flow control only -- what they guard was read or written by the tensor core or the copy
// engine, never by the other CTA's threads -- and the cluster-scope acquire costs an L1
// invalidation (CCTL.IVALL) per wait.
__device__ __forceinline__ void azb_wait_cluster(uint64_t *bar, uint32_t parity)
{
    azt_mbar_wait(bar, parity);
}

// The count of output slabs whose bulk store to global memory has COMPLETED, kept in both CTAs'
// shared memory by C's storer (chained blocks only: the next block's loads of a slab wait for it).
__device__ __forceinline__ void azb_publish(volatile uint32_t *own, uint32_t v)
{
    *own = v;
    asm volatile("st.relaxed.cluster.shared::cluster.u32 [%0], %1;" ::"r"(azb_remote((const void *)own, 0)), "r"(v) : "memory");
}

__device__ __forceinline__ void azb_wait_stored(const volatile uint32_t *cnt, uint32_t need)
{
    while (*cnt < need) asm volatile("nanosleep.u32 64;");
}

// A role's position in the chained sequence of slabs: t = pass * nslabs + j runs over all the
// passes (rings, barrier phases and the TMEM ring continue across a pass boundary; nslabs is a
// multiple of the board size, so the board row of slab t is t % n), j addresses global memory.
struct azb_pos {
    int t, j, pass;
    __device__ __forceinline__ void advance(int step, int nslabs)
    {
        t += step; j += step;
        while (nslabs > 0 && j >= nslabs) { j -= nslabs; pass++; }
    }
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(AZB_THREADS, 1)
k_resblock(const azb_params p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t rank = azb_cluster_rank();
    const bool isP = rank == 0;                                     // conv1 producer | conv2 consumer
    uint8_t *s_w = smem;                                            // this CTA's layer, 72 KB
    uint8_t *s_in = smem + AZT_WBYTES;                              // input ring: same offset in both CTAs
    uint8_t *s_res = s_in + AZB_SY * AZT_CHUNK_BYTES;               // C: residual ring
    uint8_t *s_out = isP ? s_in + AZB_SX * AZT_CHUNK_BYTES : s_res + AZB_SR * AZT_OUT_BYTES;   // staging tiles
    const int S = isP ? AZB_SX : AZB_SY, T = isP ? AZB_TP : AZB_TC;
    __shared__ uint64_t bar_w, bar_in_full[AZB_SMAX];
    __shared__ uint64_t bar_out_empty[AZB_TMAX], bar_out_done[AZB_TMAX];    // staging tiles
    __shared__ uint64_t bar_res_full[AZB_SR], bar_res_empty[AZB_SR];        // C: residual ring
    __shared__ uint64_t bar_mma_done[8];            // MMA(t) retired, by t & 7
    __shared__ uint64_t bar_blk_free[AZT_BLOCKS];   // ring block read, zeroed and free for its next output slab
    __shared__ uint64_t bar_y_free[AZB_SY];         // P: stage of C's ring consumed (arrived by C)
    __shared__ uint32_t tmem_holder;
    __shared__ volatile uint32_t s_stored;          // output slabs (index t) whose store has completed
    __shared__ __align__(16) float s_bias[AZB_MAXPASS * AZT_C];     // this CTA's layer of every pass

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        azt_mbar_init(&bar_w, 1);
        for (int i = 0; i < AZB_SMAX; i++) azt_mbar_init(&bar_in_full[i], 1);   // one bulk transfer per stage
        for (int i = 0; i < AZB_TMAX; i++) {
            azt_mbar_init(&bar_out_empty[i], 1);        // P: C's relay (the copy has landed); C: its storer
            azt_mbar_init(&bar_out_done[i], 8);         // one arrival per warp of the group that wrote the slab
        }
        for (int i = 0; i < AZB_SR; i++) {
            azt_mbar_init(&bar_res_full[i], 1);
            azt_mbar_init(&bar_res_empty[i], 8);        // the eight warps of the group that read it
        }
        for (int i = 0; i < 8; i++) azt_mbar_init(&bar_mma_done[i], 1);
        // one arrival per warp of the group that drained the block
        for (int i = 0; i < AZT_BLOCKS; i++) azt_mbar_init(&bar_blk_free[i], 8);
        for (int i = 0; i < AZB_SY; i++) azt_mbar_init(&bar_y_free[i], 1);
        s_stored = 0;
        asm volatile("fence.mbarrier_init.release.cluster;");
        // C arms every stage of its input ring for the first slab P will copy into it
        if (!isP)
            for (int i = 0; i < AZB_SY; i++) azt_mbar_expect_tx(&bar_in_full[i], AZT_OUT_BYTES);
    }
    for (int i = tid; i < p.passes * AZT_C; i += AZB_THREADS)
        s_bias[i] = p.bias[((i / AZT_C) * 2 + rank) * AZT_C + (i % AZT_C)];
    if (!isP) {
        // P only ever writes the 128 slab rows of a stage; the 8 rows in front of them are the
        // zero rows every slab is preceded by, the 8 rows behind feed masked outputs only
        for (int i = tid; i < AZB_SY * AZT_CHUNK_BYTES / 16; i += AZB_THREADS)
            reinterpret_cast<uint4 *>(s_in)[i] = make_uint4(0u, 0u, 0u, 0u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(azt_smem(&tmem_holder)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = tmem_holder;

    // this cluster's contiguous range of groups -> slabs [q0, q0 + nslabs) of every pass; NT slabs
    // in all, t = pass * nslabs + j; board row y = t % n
    const int n = p.n;
    const long long cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
    // packed leaves: the batch holds *live boards, known only on the device; the grid was sized
    // for p.groups, clusters left without a group fall through every role
    long long groups = p.groups;
    if (p.live != nullptr) {
        const long long lg = ((long long)*p.live + p.bpg - 1) / p.bpg;
        groups = lg < groups ? lg : groups;
    }
    const long long g0 = groups * cid / ncl, g1 = groups * (cid + 1) / ncl;
    const long long q0 = g0 * n;
    const int nslabs = (int)((g1 - g0) * n);
    const int NT = nslabs * p.passes;
#define AZB_RING(u) ((8 - ((u) & 7)) & 7)

    if (warp < 16) {
        // zero the whole accumulator ring once: every MMA accumulates
        const uint32_t tq = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        for (int c = (warp >> 2) * 16; c < 512; c += 64) azt_tmem_zero16(tq + c);
        asm volatile("tcgen05.wait::st.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    // both CTAs' barriers are initialised (and C's ring zeroed) before either touches the other's
    azb_cluster_sync();

    if (NT == 0) {
        // packed leaves: fewer live groups than clusters -- this one has nothing to do (both of its
        // CTAs agree); it still takes part in the two cluster barriers and frees its TMEM
    } else if (warp == 20) {
        // ------------------------------------------------------------ storer --
        // A bulk store takes ~1000 cycles to read its 16 KB tile, and bulk groups are per
        // thread: one storer thread that waits for each store's read before it hands the tile
        // back caps the pipeline AROUND the MMAs at ~1200 cycles per slab (measured with the MMAs
        // switched off); with the MMAs running the kernel is bound elsewhere.
        if (isP && lane == 0) {
            // P: finished y slab: staging tile -> rows 8..135 of stage st of C's input ring
            for (int t = 0; t < NT; t++) {
                const int sb = t % AZB_TP, st = t % AZB_SY;
                azt_mbar_wait(&bar_out_done[sb], (t / AZB_TP) & 1);
                if (t >= AZB_SY) azb_wait_cluster(&bar_y_free[st], ((t / AZB_SY) & 1) ^ 1);
                azb_bulk_s2s(azb_remote(s_in + st * AZT_CHUNK_BYTES + 8 * AZT_ROW, 1),
                             s_out + sb * AZT_OUT_BYTES, AZT_OUT_BYTES, azb_remote(&bar_in_full[st], 1));
            }
        } else if (lane == 0) {
            // C: finished output slab -> global memory, in place
            azb_pos at = {0, 0, 0};
            for (; at.t < NT; at.advance(1, nslabs)) {
                const int sb = at.t % AZB_TC;
                azt_mbar_wait(&bar_out_done[sb], (at.t / AZB_TC) & 1);
                azt_bulk_s2g(p.x + (size_t)(AZT_HALO + (q0 + at.j) * 128) * AZT_ROW, s_out + sb * AZT_OUT_BYTES,
                             AZT_OUT_BYTES);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                // hand the tile back as soon as the store has READ it (the write to global
                // memory goes on): each epilogue group has one tile
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                azt_mbar_arrive(&bar_out_empty[sb]);
                if (p.passes > 1) {
                    // chained blocks: the next pass loads these slabs again (P as its input, C as
                    // its residual) once their stores have COMPLETED.  All stores but this one
                    // have (the last slab of a pass: this one too); say so in both CTAs.
                    if (at.j + 1 == nslabs) {
                        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
                        azb_publish(&s_stored, (uint32_t)at.t + 1u);
                    } else {
                        asm volatile("cp.async.bulk.wait_group 1;" ::: "memory");
                        azb_publish(&s_stored, (uint32_t)at.t);
                    }
                }
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
    } else if (warp == 19) {
        // ------------------------ relay (C, lane 0) / weights (both, lane 1) --
        if (lane == 1) {
            // both CTAs: this layer's weights, pass after pass.  The thread follows EVERY slab's
            // "MMA retired" barrier in order (a parity wait is only sound one phase away), and
            // loads the next pass's weights when the last slab of a pass has retired.
            const uint8_t *w = p.w + (size_t)rank * AZT_WBYTES;
            for (int pass = 0; pass < p.passes && NT > 0; pass++) {
                if (pass > 0)
                    for (int t = (pass - 1) * nslabs; t < pass * nslabs; t++)
                        azt_mbar_wait(&bar_mma_done[t & 7], (t >> 3) & 1);
                azt_mbar_expect_tx(&bar_w, AZT_WBYTES);
                for (int tp = 0; tp < 9; tp++)
                    azt_bulk_g2s(s_w + tp * 8192, w + (size_t)(pass * 2) * AZT_WBYTES + tp * 8192, 8192, &bar_w);
            }
        } else if (!isP && lane == 0) {
            for (int t = 0; t <= NT; t++) {
                if (t < NT) {
                    // slab t has landed in C: P's staging tile that held it may be rewritten
                    azb_wait_cluster(&bar_in_full[t % AZB_SY], (t / AZB_SY) & 1);
                    azb_remote_arrive(azb_remote(&bar_out_empty[t % AZB_TP], 0));
                }
                if (t >= 1 && t - 1 + AZB_SY < NT) {
                    // MMA2(t-1) has read its stage: arm it for its next slab, then let P copy that in
                    const int k = t - 1;
                    azt_mbar_wait(&bar_mma_done[k & 7], (k >> 3) & 1);
                    azt_mbar_expect_tx(&bar_in_full[k % AZB_SY], AZT_OUT_BYTES);
                    azb_remote_arrive(azb_remote(&bar_y_free[k % AZB_SY], 0));
                }
            }
        }
    } else if (warp == 18) {
        // ------------------------------------------------------------ loader --
        if (lane == 0 && isP) {
            azb_pos at = {0, 0, 0};
            for (; at.t < NT; at.advance(1, nslabs)) {
                const int st = at.t % AZB_SX;
                // the stage is free once the MMAs of the slab that used it last have retired
                if (at.t >= AZB_SX) azt_mbar_wait(&bar_mma_done[(at.t - AZB_SX) & 7], ((at.t - AZB_SX) >> 3) & 1);
                // chained blocks: the slab is the previous pass's output
                if (at.pass > 0) azb_wait_stored(&s_stored, (uint32_t)(at.t - nslabs) + 1u);
                // slab rows plus 8 rows on each side: global rows [128 q, 128 q + 144)
                azt_mbar_expect_tx(&bar_in_full[st], AZT_CHUNK_BYTES);
                azt_bulk_g2s(s_in + st * AZT_CHUNK_BYTES, p.x + (size_t)((q0 + at.j) * 128) * AZT_ROW,
                             AZT_CHUNK_BYTES, &bar_in_full[st]);
            }
        } else if (lane == 0) {
            // C: the residual: the block's own input slab, again (L2: P has just read it)
            azb_pos at = {0, 0, 0};
            for (; at.t < NT; at.advance(1, nslabs)) {
                const int sr = at.t % AZB_SR;
                azt_mbar_wait(&bar_res_empty[sr], ((at.t / AZB_SR) & 1) ^ 1);
                // chained blocks: the slab is this CTA's own output of the previous pass
                if (at.pass > 0) azb_wait_stored(&s_stored, (uint32_t)(at.t - nslabs) + 1u);
                azt_mbar_expect_tx(&bar_res_full[sr], AZT_OUT_BYTES);
                azt_bulk_g2s(s_res + sr * AZT_OUT_BYTES, p.x + (size_t)(AZT_HALO + (q0 + at.j) * 128) * AZT_ROW,
                             AZT_OUT_BYTES, &bar_res_full[sr]);
            }
        }
    } else if (warp >= 16) {
        // -------------------------------------------------- MMA issuers --
        // Warp 16 issues the even slabs, warp 17 the odd ones (az_tower.cuh).  The turn passes
        // through named barriers 3 (-> even) and 4 (-> odd).
        const int w = warp - 16;
        const uint64_t db_base = azt_desc(azt_smem(s_w));
        if (w == 1 && NT > 0) asm volatile("bar.arrive 3, 64;" ::: "memory");   // slab 0 has the first turn
        int wpass = -1;                     // pass whose weights this warp has waited for
        azb_pos at = {w, w, 0};
        at.advance(0, nslabs);
        for (int y = w % n; at.t < NT; at.advance(2, nslabs), y = (y + 2) % n) {
            const int t = at.t, st = t % S;
            // input slab t feeds output slabs t+1 (dy 0), t (dy 1), t-1 (dy 2) of the same group
            const int dy0 = y + 1 < n ? 0 : 1, dy1 = y > 0 ? 2 : 1;
            const int top = t + 1 - dy0;
            // highest output slab entered by the slabs before this one
            const int entered = t == 0 ? -1 : (y == 0 ? t - 1 : t);
            azb_wait_cluster(&bar_in_full[st], (t / S) & 1);
            // this pass's weights (the other warp's MMAs of the last pass retire before they are replaced)
            while (wpass < at.pass) { wpass++; azt_mbar_wait(&bar_w, wpass & 1); }
            // a block entered for a new output slab u: its previous tenant u-8 must have been retired
            for (int u = entered + 1; u <= top; u++)
                if (u >= 8) azt_mbar_wait(&bar_blk_free[AZB_RING(u)], ((u >> 3) - 1) & 1);
            const int blk = AZB_RING(top), nb = dy1 - dy0 + 1;
            const int first = nb < 8 - blk ? nb : 8 - blk, second = nb - first;     // split where the ring wraps
            const uint32_t d0 = tmem + blk * 64, i0 = AZT_IDESC(first), i1 = AZT_IDESC(second);
            // descriptors advance in 16-byte units: one row = 8, one K step (32 B) = 2
            const uint64_t da0 = azt_desc(azt_smem(s_in + st * AZT_CHUNK_BYTES) + 7 * AZT_ROW);    // row l-1 of the slab
            const uint64_t db0 = db_base + (uint64_t)(dy0 * 64 * (AZT_ROW / 16));
            const uint64_t db1 = db0 + (uint64_t)(first * 64 * (AZT_ROW / 16));
            // take the turn: the other warp has issued slab t-1
            if (w == 0) asm volatile("bar.sync 3, 64;" ::: "memory");
            else asm volatile("bar.sync 4, 64;" ::: "memory");
            asm volatile("tcgen05.fence::after_thread_sync;");
            if (azt_elect()) {
                if (second == 0) {
#pragma unroll
                    for (int dx = 0; dx < 3; dx++)
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            azt_mma(d0, da0 + (dx * 8 + k * 2), db0 + (dx * 192 * 8 + k * 2), i0);
                } else {
                    // one accumulator range after the other (tools/probe/umma_gap.cu)
#pragma unroll
                    for (int dx = 0; dx < 3; dx++)
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            azt_mma(d0, da0 + (dx * 8 + k * 2), db0 + (dx * 192 * 8 + k * 2), i0);
#pragma unroll
                    for (int dx = 0; dx < 3; dx++)
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            azt_mma(tmem, da0 + (dx * 8 + k * 2), db1 + (dx * 192 * 8 + k * 2), i1);
                }
                // one commit per slab: output slabs wait for it, and so does the input stage
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                             ::"r"(azt_smem(&bar_mma_done[t & 7])) : "memory");
            }
            __syncwarp();
            asm volatile("tcgen05.fence::before_thread_sync;");
            if (t + 1 < NT) {
                if (w == 0) asm volatile("bar.arrive 4, 64;" ::: "memory");
                else asm volatile("bar.arrive 3, 64;" ::: "memory");
            }
        }
    } else {
        // ----------------------------------------------------- epilogue --
        // group = warp >> 3 takes the output slabs t = group (mod 2); inside a group a warp
        // owns 32 channels (half) of the 32 rows its TMEM lane quadrant holds:
        // thread = TMEM lane = row l of the slab
        const int grp = warp >> 3, half = (warp >> 2) & 1, wq = warp & 3;
        const int l = wq * 32 + lane;
        const bool real = l < p.bpg * (n + 1) && (l % (n + 1)) != n;    // not a pad cell
        const uint32_t keep = real ? 0xffffffffu : 0u;
        const int sw = l & 7;                                       // == R & 7 (8 + 128 q + l)
        azb_pos at = {grp, grp, 0};
        at.advance(0, nslabs);
        for (int y = grp % n; at.t < NT; at.advance(2, nslabs), y = (y + 2) % n) {
            const int t = at.t, sb = t % T;
            const float *bias = s_bias + at.pass * AZT_C;
            uint4 *srow = reinterpret_cast<uint4 *>(s_out + sb * AZT_OUT_BYTES + l * AZT_ROW);
            uint4 rv[4];
            if (!isP) {
                // this thread's row and channels of the residual slab, from the bulk-loaded ring
                const int sr = t % AZB_SR;
                azt_mbar_wait(&bar_res_full[sr], (t / AZB_SR) & 1);
                const uint4 *rrow = reinterpret_cast<const uint4 *>(s_res + sr * AZT_OUT_BYTES + l * AZT_ROW);
#pragma unroll
                for (int c = 0; c < 4; c++) rv[c] = rrow[(half * 4 + c) ^ sw];
                // The release below hands the stage to the NEXT BULK LOAD (async proxy).  An
                // mbarrier arrive does not wait for the shared-memory loads issued before it:
                // without this the arrive overtook them and slow warps read the slab that was
                // loaded three slabs later (~2 % of the rows; profiles/r02_fused_block.txt).
                // Consuming the loaded registers in a warp vote makes every lane's loads return
                // before lane 0 can arrive.  (fence.proxy.async here is the other cure and costs
                // 4 %; __threadfence_block is not one.)
                if (__any_sync(0xffffffffu, (rv[0].x ^ rv[1].y ^ rv[2].z ^ rv[3].w) == 0x7fc1a55eu &&
                                                (rv[0].y ^ rv[1].x) == 0x5ea1c0deu && rv[2].x == 0xfeedbeefu))
                    asm volatile("nanosleep.u32 1;");
                __syncwarp();
                if (lane == 0) azt_mbar_arrive(&bar_res_empty[sr]);
            }
            // the staging tile must have been drained by the copy / store that used it last
            azb_wait_cluster(&bar_out_empty[sb], ((t / T) & 1) ^ 1);
            // output slab t is complete once MMA(t+1) retired (MMA(t) for the last board row)
            const int last = y + 1 < n ? t + 1 : t;
            azt_mbar_wait(&bar_mma_done[last & 7], (last >> 3) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;");
            const int blk = AZB_RING(t);
            const uint32_t ta = tmem + ((uint32_t)(wq * 32) << 16) + (uint32_t)blk * 64u + (uint32_t)half * 32u;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                uint32_t acc[16];
                AZT_TMEM_LD16(acc, ta + h * 16);
                asm volatile("tcgen05.wait::ld.sync.aligned;");
                azt_tmem_zero16(ta + h * 16);       // retire: zero for the block's next output slab
#pragma unroll
                for (int g = 0; g < 2; g++) {
                    const int c8 = half * 4 + h * 2 + g;            // 8-channel chunk of the row
                    const float4 b0 = *reinterpret_cast<const float4 *>(&bias[c8 * 8]);
                    const float4 b1 = *reinterpret_cast<const float4 *>(&bias[c8 * 8 + 4]);
                    float f[8];
                    f[0] = __uint_as_float(acc[g * 8 + 0]) + b0.x; f[1] = __uint_as_float(acc[g * 8 + 1]) + b0.y;
                    f[2] = __uint_as_float(acc[g * 8 + 2]) + b0.z; f[3] = __uint_as_float(acc[g * 8 + 3]) + b0.w;
                    f[4] = __uint_as_float(acc[g * 8 + 4]) + b1.x; f[5] = __uint_as_float(acc[g * 8 + 5]) + b1.y;
                    f[6] = __uint_as_float(acc[g * 8 + 6]) + b1.z; f[7] = __uint_as_float(acc[g * 8 + 7]) + b1.w;
                    if (!isP) {
                        const uint4 r = rv[h * 2 + g];
                        const uint32_t rw[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            f[2 * q] += __uint_as_float(rw[q] << 16);
                            f[2 * q + 1] += __uint_as_float(rw[q] & 0xffff0000u);
                        }
                    }
                    uint32_t ow[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        ow[q] = azt_relu_bf16x2(f[2 * q], f[2 * q + 1]) & keep;
                    }
                    // chunk c8 of the row, at its swizzled place in the staging tile
                    srow[c8 ^ sw] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
                }
            }
            // hand the ring block back
            asm volatile("tcgen05.wait::st.sync.aligned;");
            asm volatile("tcgen05.fence::before_thread_sync;");
            __syncwarp();
            if (lane == 0) azt_mbar_arrive(&bar_blk_free[blk]);
            // staging tile complete: the storer sends it on (the copy engine, async proxy, reads it)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) azt_mbar_arrive(&bar_out_done[sb]);
        }
    }
#undef AZB_RING
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    // neither CTA may leave while the other can still reach into its shared memory
    azb_cluster_sync();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
}
