// bp_node_kernels.cu -- frame streams in the node-state formulation of flooding BP on the BEC (sm_100a).
//
// From the all-erased start the messages of flooding BP on the BEC are monotone, and the a-posteriori erased set after
// iteration t is a function of the erased set after iteration t-1 alone ("parallel peeling"):
//
//     x_v(t) = x_v(t-1)  AND NOT  (some CN of v has v as its only erased neighbour in x(t-1))
//
// (an extrinsic message that the message-passing decoder would still hold back can only concern a VN that is already
// known, see DESIGN.md section 4).  The erased set -- hence the residual erasures, the per-frame iteration count under the
// reference's stall rule (NumErasures == NumErasuresPrec, BP_FULL.c:1046-1066), the error counts and the expurgation
// inputs -- is bit-identical to decodeBP's at every iteration; tests/test_stream_gpu.py holds it against the message
// kernels (themselves checked against the oracle and the compiled reference) and tests/test_full_size_ref_gpu.py against
// the compiled reference at the benchmarked size.  What the formulation does not carry are the messages, so the trajectory
// mode (deg_1_iter, BP_TRAJ.c:935-979) stays on the message kernels (bp_kernels.cu / bp_wave_kernels.cu).
//
// ONE launch per flooding iteration.  State per graph: two planes [n][chunks] (1 bit per VN and frame) that alternate as
// "read" (the state after the previous iteration, which every CN of the sweep reads: that is the flooding schedule) and
// "write" (where resolved bits are cleared).  Round 1 made the planes equal again with a sequential pass over the whole
// plane after every sweep (41 % of an iteration: 69 MB streamed to move the ~6 % of rows that had changed).  Now every
// warp of the sweep logs its resolutions -- (32-bit word of the plane, bit) -- into a private region, and the SAME warp
// of the NEXT launch replays its region on that launch's write plane before it sweeps.  Clearing is commutative
// (red.and), so the replay needs no ordering against the new resolutions, and nothing reads the write plane until the
// launch after.  A region that overflows (the dense first iteration of a stream) raises a flag and the next launch
// catches up with one full pass, so the lists never have to be sized for the worst case.
//
// "An erased VN is left" is no longer tracked per iteration either (it was the other reason for the full pass).  A frame
// that resolves its last VN in iteration t is seen to stop in t+1 ("nothing resolved"); the harvest, which counts the
// residual erasures of every stopped frame anyway, takes that extra iteration off again (lazy_success).  A frame that
// stalls with erasures left stops in the iteration the reference stops in.  Iteration counts, residuals and every
// derived statistic stay bit-identical; the ride-along iteration costs about 1/350 of the work.
//
// Useful work is still accounted as the reference's: 2E edge updates per frame-iteration.
#include "common.cuh"

namespace scldpc {

// ------------------------------------------------------------------------------------------------------------
// one flooding iteration: replay, check-node sweep, end of the iteration (last block)
// ------------------------------------------------------------------------------------------------------------
// CN sweep: a CN with exactly one erased neighbour in the read plane resolves it -- the bit is cleared in the write plane.
// Resolutions are sparse (a VN is resolved once per frame; about 0.5 per thread and trip), so the scatter is a short divergent
// loop; the index of the neighbour to clear is carried in bit planes next to the saturating count.
// The sweep is bound by L2 latency and instruction issue, not by HBM (DESIGN.md section 4).
// M is the stream mode (common.cuh); SM_PLAIN streams run unlimited BP and nothing more.
// SM_CAPPED (streams with an iteration cap): a frame that hit the cap is not at a fixed point, so its bits must not be cleared
// while it waits for the harvest -- the resolutions are masked with the frames still iterating.
// SM_CKPT (streams with checkpoints, capped as well): a frame that reaches its next checkpoint caps[lane_ck] without stopping
// in that iteration pauses -- it leaves active for pause_mask, not done_mask -- and the harvest records its statistics and
// puts it back into active.  A paused lane is masked like a capped one, and its lane_iter does not advance.
// SM_HEAD (streams with stopping-set records, unlimited): the unscanned head of simulate_sc_ldpc with is_bounded = False, per
// lane.  A CN below cn_dis_lim that starts a frame with exactly one erased neighbour never resolves it (bpw_iter_kernel<.,.,HEAD>);
// "starts" is the frame's first iteration, the launch after the harvest that armed its lane (head_arm), so the cn_dis bits of
// the armed lanes are set there and every other lane keeps its own.
template <int DV, int DC, StreamMode M>
__global__ void __launch_bounds__(32 * NS_WARPS, 4) ns_iter_kernel(BpParams p)
{
    constexpr bool CAPPED = M == SM_CAPPED || M == SM_CKPT;     // resolutions masked with the frames still iterating
    static_assert(DC <= 16, "neighbour index is encoded in four bit planes");
    pdl_wait_then_release();
    const int g = graph_of(p, blockIdx.y);
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ u64 s_new[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (threadIdx.x < SCLDPC_MAX_WORDS) s_new[threadIdx.x] = 0;
    __syncthreads();
    const int ch = p.chunks;                                    // row stride of the planes
    // chunks the graph's live frames occupy: all of them until the tail of the stream, where the lane compaction (below) moves
    // the frames still decoding into the lowest chunks and the sweep spreads its threads over those chunks only
    const int cs = ld_cg(p.gshift + g), chn = 1 << cs;
    const int k = threadIdx.x & (chn - 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int par = p.iter & 1;
    const size_t plane = (size_t)g * p.n * ch;
    const u128 *__restrict__ rd = (par ? p.xb : p.x) + plane;
    u128 *__restrict__ wr = (par ? p.x : p.xb) + plane;
    unsigned *__restrict__ wr32 = reinterpret_cast<unsigned *>(wr);
    const int RW = p.nl_rw;
    const int rid = blockIdx.x * NS_WARPS + warp;

    // ---- the write plane catches up with the previous iteration ----
    if (ld_cg(p.nl_ovf + g * 2 + (par ^ 1))) ns_catch_up(rd, wr, 0, p.n << p.chunk_shift);
    else ns_replay_region(p, g, par ^ 1, wr32, rid, false);

    // ---- check-node sweep ----
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const bool lane_work = nz(act);                             // a thread keeps its chunk
    const u128 *__restrict__ rdk = rd + k;
    const int32_t *__restrict__ cn_row = p.cn_row + (size_t)g * p.nk * DC;
    uint2 *__restrict__ reg = p.nl_list + ((size_t)(g * 2 + par) * RW + rid) * p.nl_stride;
    const int items = p.c1 << cs;                               // CNs >= c1 (tail of a truncated code) are never swept
    const int stride = gridDim.x * blockDim.x;
    int wcount = 0;                                             // entries this warp has logged (warp-uniform)
    u128 acc_new = zero128();
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < items; base += stride) {
        const int idx = base + lane;
        u128 res = zero128(), b0 = zero128(), b1 = zero128(), b2 = zero128(), b3 = zero128();
        const int32_t *row = cn_row + (size_t)(idx >> cs) * DC;
        if (lane_work && idx < items) {
            int e[DC];
            load_row<DC>(row, e);
            u128 in[DC];
#pragma unroll
            for (int j = 0; j < DC; j++) in[j] = ld_stream(rdk + (unsigned)e[j]);
            // saturating count of erased neighbours (one / two planes) and, in bit planes b0..b3, the index j of an erased
            // neighbour -- exact where it is needed, i.e. in the frames with exactly one
            u128 one = zero128(), tw = zero128();
#pragma unroll
            for (int j = 0; j < DC; j++) {
                tw |= one & in[j];
                one |= in[j];
                if (j & 1) b0 |= in[j];
                if (j & 2) b1 |= in[j];
                if (j & 4) b2 |= in[j];
                if (j & 8) b3 |= in[j];
            }
            res = one & ~tw;                                    // frames in which exactly one neighbour of c is erased
            if (CAPPED) res &= act;
            if (M == SM_HEAD && (idx >> cs) < p.cn_dis_lim) {
                // one 64-bit half at a time, with 32-bit word offsets (the plane offsets are below 2^32, see capi.cu): the u128
                // merge with 64-bit pointers spilled the (4,12) and (3,9) sweeps
                const unsigned dw = 2u * (((unsigned)g * (unsigned)p.cn_dis_lim + (unsigned)(idx >> cs)) * (unsigned)ch + (unsigned)k);
                const unsigned aw = (unsigned)g * (unsigned)p.W + 2u * (unsigned)k;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    u64 &r = h ? res.y : res.x;
                    u64 *dp = reinterpret_cast<u64 *>(p.cn_dis) + dw + h;
                    const u64 dis = *dp;
                    const u64 arm = p.head_arm ? p.arm_mask[aw + h] : 0ull;
                    const u64 nd = (r & arm) | (dis & ~arm);
                    if (nd != dis) *dp = nd;
                    r &= ~nd;
                }
            }
        }
        if (__ballot_sync(0xffffffffu, nz(res)) == 0u) continue;
        // slots of this trip's resolutions in the warp's region: exclusive prefix sum of the per-thread counts
        const int c = __popcll(res.x) + __popcll(res.y);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        int slot = wcount + incl - c;
        wcount += __shfl_sync(0xffffffffu, incl, 31);
        if (c) {
            acc_new |= res;
            const unsigned rw[4] = {(unsigned)res.x, (unsigned)(res.x >> 32), (unsigned)res.y, (unsigned)(res.y >> 32)};
            const unsigned w0[4] = {(unsigned)b0.x, (unsigned)(b0.x >> 32), (unsigned)b0.y, (unsigned)(b0.y >> 32)};
            const unsigned w1[4] = {(unsigned)b1.x, (unsigned)(b1.x >> 32), (unsigned)b1.y, (unsigned)(b1.y >> 32)};
            const unsigned w2[4] = {(unsigned)b2.x, (unsigned)(b2.x >> 32), (unsigned)b2.y, (unsigned)(b2.y >> 32)};
            const unsigned w3[4] = {(unsigned)b3.x, (unsigned)(b3.x >> 32), (unsigned)b3.y, (unsigned)(b3.y >> 32)};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                unsigned m = rw[q];
                while (m) {
                    const int b = __ffs((int)m) - 1;
                    m &= m - 1;
                    int j = ((w0[q] >> b) & 1u) | (((w1[q] >> b) & 1u) << 1) | (((w2[q] >> b) & 1u) << 2);
                    if (DC > 8) j |= ((w3[q] >> b) & 1u) << 3;
                    const unsigned widx = 4u * ((unsigned)__ldg(row + j) + (unsigned)k) + (unsigned)q;   // L1 hit
                    red_and(wr32 + widx, ~(1u << b));
                    if (slot < p.nl_cap) st_cg_u2(reg + slot, make_uint2(widx, 1u << b));
                    slot++;
                }
            }
        }
    }
    if (lane == 0) {
        p.nl_cnt[(size_t)(g * 2 + par) * RW + rid] = wcount < p.nl_cap ? wcount : p.nl_cap;
        if (wcount > p.nl_cap) p.nl_ovf[g * 2 + par] = 1;
    }
    acc_new = warp_or_same_chunk(acc_new, chn);
    if (lane < chn) {
        if (acc_new.x) atomicOr(&s_new[2 * k], acc_new.x);
        if (acc_new.y) atomicOr(&s_new[2 * k + 1], acc_new.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_new[w] & ~ld_cg(p.any_new + g * p.W + w)) atomicOr(p.any_new + g * p.W + w, s_new[w]);
    }
    __threadfence();                                            // list counts, overflow flag, any_new: read by the last block / next launch
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- end of the iteration for graph g ----
    __shared__ u64 s_act[SCLDPC_MAX_WORDS], s_cap[SCLDPC_MAX_WORDS];
    __shared__ u64 s_ck[M == SM_CKPT ? SCLDPC_MAX_WORDS : 1];
    const int W = p.W;
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        s_act[w] = p.active[g * W + w]; s_cap[w] = 0;
        if (M == SM_CKPT) s_ck[w] = 0;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_act[w] >> b) & 1ull) {
            const int li = p.lane_iter[g * p.lanes + l] + 1;
            p.lane_iter[g * p.lanes + l] = li;
            if (CAPPED && li >= p.stream_cap) atomicOr(reinterpret_cast<unsigned long long *>(&s_cap[w]), 1ull << b);   // while (iter < MaxNumIt)
            else if (M == SM_CKPT) {
                const int ck = p.lane_ck[g * p.lanes + l];
                if (ck < p.n_caps - 1 && li >= p.caps[ck]) atomicOr(reinterpret_cast<unsigned long long *>(&s_ck[w]), 1ull << b);
            }
        }
    }
    __syncthreads();
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        const u64 a = s_act[w];
        // lanes armed by the last harvest run their first iteration: NumErasuresPrec = n, so it makes "progress" iff the
        // channel left some VN known (first_new)
        const u64 nw = ld_cg(p.any_new + g * W + w) | ld_cg(p.first_new + g * W + w);
        const u64 stop = a & (~nw | s_cap[w]);                  // NumErasures == NumErasuresPrec (or == 0, one iteration late) || cap
        if (M == SM_CKPT) {
            const u64 pause = s_ck[w] & ~stop;                  // a frame that stops at a checkpoint stops
            p.active[g * W + w] = a & ~stop & ~pause;
            if (pause) p.pause_mask[g * W + w] |= pause;
        } else
            p.active[g * W + w] = a & ~stop;
        p.done_mask[g * W + w] |= stop;
        p.noprog[g * W + w] |= a & ~nw;
        p.any_new[g * W + w] = 0;
        p.first_new[g * W + w] = 0;
    }
    if (threadIdx.x == 0) {
        p.nl_ovf[g * 2 + (par ^ 1)] = 0;                        // consumed by every block of this launch
        p.ticket[g] = 0;
    }
}

// Before a harvest: the plane the last iteration read catches up, so both planes are equal and the lists are empty
// (lanes are re-armed with new frames right after; a replay after that would clear bits of the new frames).
__global__ void __launch_bounds__(32 * NS_WARPS) ns_settle_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y);
    if (ld_cg(p.alive + g) == 0) return;
    const int par_prev = (p.iter & 1) ^ 1;                      // p.iter: the iteration that runs next
    const size_t plane = (size_t)g * p.n * p.chunks;
    const u128 *rd = ((p.iter & 1) ? p.xb : p.x) + plane;       // complete: the last iteration wrote it
    u128 *wr = ((p.iter & 1) ? p.x : p.xb) + plane;
    __shared__ int s_ovf;
    if (threadIdx.x == 0) s_ovf = ld_cg(p.nl_ovf + g * 2 + par_prev);
    __syncthreads();
    if (s_ovf) ns_catch_up(rd, wr, 0, p.n << p.chunk_shift);
    else ns_replay_region(p, g, par_prev, reinterpret_cast<unsigned *>(wr), blockIdx.x * NS_WARPS + (threadIdx.x >> 5), true);
}
__global__ void ns_settle_done_kernel(BpParams p)
{
    const int RW = p.nl_rw;
    const int g = graph_of(p, blockIdx.x), par_prev = (p.iter & 1) ^ 1;
    if (ld_cg(p.nl_ovf + g * 2 + par_prev) == 0) return;
    for (int i = threadIdx.x; i < RW; i += blockDim.x) p.nl_cnt[(size_t)(g * 2 + par_prev) * RW + i] = 0;
    if (threadIdx.x == 0) p.nl_ovf[g * 2 + par_prev] = 0;
}

// After a harvest: the freed lanes take their new frames.  The erased set starts as the channel's (Lji = channel value on
// every edge, BP_FULL.c:913-917), written to both planes; the lanes iterate from the next launch on.
//
// The harvest hands out consecutive frame ids in ascending lane order, so the armed lanes of a graph are one run of frame ids
// [f0, f0+A) and one Philox call -- four frames of one VN -- serves four armed lanes wherever they sit in the row.  A block takes
// tiles of ARM_ROWS VN rows: phase 1 spreads (row, Philox block) pairs over the threads and ORs the erased frames into a shared
// copy of the rows' armed bits (at most ceil(A/4)+1 calls per VN, against one call per armed lane and 128-lane chunk when every
// thread drew the lanes of its own chunk: the kernel was 7.8 % of the benchmarked step, profiles/r02e); phase 2 merges the tile
// into both planes with coalesced 16-byte accesses.
#define ARM_ROWS 128
__global__ void __launch_bounds__(256, 4) ns_arm_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y);
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ u64 s_first[SCLDPC_MAX_WORDS], s_armw[SCLDPC_MAX_WORDS];
    __shared__ int s_rank[SCLDPC_MAX_WORDS + 1];
    __shared__ unsigned short s_lane[SCLDPC_MAX_LANES];
    __shared__ unsigned s_bits[ARM_ROWS * 2 * SCLDPC_MAX_WORDS];
    const int W = p.W, ch = p.chunks, RWORDS = 2 * W;           // 32-bit words per plane row
    if (threadIdx.x < SCLDPC_MAX_WORDS) {
        s_first[threadIdx.x] = 0;
        s_armw[threadIdx.x] = threadIdx.x < W ? p.arm_mask[g * W + threadIdx.x] : 0ull;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int r = 0;
        for (int w = 0; w < W; w++) { s_rank[w] = r; r += __popcll(s_armw[w]); }
        s_rank[W] = r;
    }
    __syncthreads();
    const int A = s_rank[W];
    if (A == 0) return;
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_armw[w] >> b) & 1ull) s_lane[s_rank[w] + __popcll(s_armw[w] & ((1ull << b) - 1ull))] = (unsigned short)l;
    }
    __syncthreads();
    const uint32_t f0 = (uint32_t)p.lane_frame[g * p.lanes + s_lane[0]];
    const uint32_t blk0 = f0 >> 2;
    const int nb = (int)(((f0 + (uint32_t)A - 1u) >> 2) - blk0) + 1;
    const int k = threadIdx.x & (ch - 1);
    const u128 arm = make_u128(s_armw[2 * k], s_armw[2 * k + 1]);
    u128 acc_first = zero128();
    u128 *__restrict__ x = p.x + (size_t)g * p.n * ch;
    u128 *__restrict__ xb = p.xb + (size_t)g * p.n * ch;
    const u64 thr = p.thr[g];
    const uint64_t gid = p.first_graph + (uint64_t)g;
    const uint32_t k0 = (uint32_t)p.seed ^ 0x6368616Eu, k1 = (uint32_t)(p.seed >> 32);
    for (int row0 = blockIdx.x * ARM_ROWS; row0 < p.n; row0 += gridDim.x * ARM_ROWS) {
        const int rows = min(ARM_ROWS, p.n - row0);
        for (int i = threadIdx.x; i < rows * RWORDS; i += blockDim.x) s_bits[i] = 0u;
        __syncthreads();
        // phase 1: channel draws, one Philox call per (VN, block of four frame ids)
        for (int item = threadIdx.x; item < rows * nb; item += blockDim.x) {
            const int vl = item / nb, j = item - vl * nb;
            const int v = row0 + vl;
            if (p.known && (v % p.vns_pos) < p.known[v / p.vns_pos]) continue;     // doped: known whatever the channel says
            uint32_t r4[4];
            philox4x32_10((uint32_t)v, blk0 + (uint32_t)j, (uint32_t)gid, (uint32_t)(gid >> 32), k0, k1, r4);
#pragma unroll
            for (int s = 0; s < 4; s++) {
                const int i = (int)(4u * (blk0 + (uint32_t)j) + (uint32_t)s - f0);
                if (i >= 0 && i < A && (u64)r4[s] < thr) {
                    const int l = s_lane[i];
                    atomicOr(&s_bits[vl * RWORDS + (l >> 5)], 1u << (l & 31));
                }
            }
        }
        __syncthreads();
        // phase 2: the armed lanes of both planes take the new frames' channel bits
        if (nz(arm))
            for (int i = threadIdx.x; i < rows << p.chunk_shift; i += blockDim.x) {   // i % ch == k: blockDim is a multiple of ch
                const unsigned *sb = s_bits + (i >> p.chunk_shift) * RWORDS + 4 * k;
                const u128 cw = make_u128((u64)sb[0] | ((u64)sb[1] << 32), (u64)sb[2] | ((u64)sb[3] << 32));
                const size_t idx = ((size_t)row0 << p.chunk_shift) + i;
                const u128 xo = x[idx];
                const u128 xn = sel(arm, cw, xo);
                if (neq(xn, xo)) { x[idx] = xn; xb[idx] = xn; }
                acc_first |= ~cw & arm;
            }
        __syncthreads();
    }
    acc_first = warp_or_same_chunk(acc_first, ch);
    if ((threadIdx.x & 31) < ch) {
        if (acc_first.x) atomicOr(&s_first[2 * k], acc_first.x);
        if (acc_first.y) atomicOr(&s_first[2 * k + 1], acc_first.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_first[w] & ~ld_cg(p.first_new + g * p.W + w)) atomicOr(p.first_new + g * p.W + w, s_first[w]);
    }
}

// ------------------------------------------------------------------------------------------------------------
// lane compaction in the tail of a stream
// ------------------------------------------------------------------------------------------------------------
// Once a graph has handed out its last frame, lanes only fall idle: the sweep keeps paying for every 128-lane chunk that
// still holds one live frame, and the slowest frames (the ones that stall, twice the iterations of the others) are spread
// over all chunks -- about 1000 of the 14 500 iterations of the benchmarked eps = 0.49 graph run with a few dozen live frames
// at the full price.  After a harvest that armed nothing, when the live frames fit into half the chunks in use, they move to
// the lowest lanes: a frame's whole decoder state is its bit column in the (equal, settled) planes plus lane_frame and
// lane_iter (and lane_ck in a stream with checkpoints, whose paused frames the harvest has just put back into active, and the
// cn_dis rows in a stream with an unscanned head), so the move is one pass over the plane; gshift[g] then tells ns_iter_kernel to spread its threads over the occupied chunks only.
// Frame results are stored under the frame id, so nothing downstream sees the lane change.
__global__ void ns_compact_plan_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.x), W = p.W;
    __shared__ u64 s_act[SCLDPC_MAX_WORDS];
    __shared__ int s_rank[SCLDPC_MAX_WORDS + 1], s_go;
    __shared__ int s_fr[SCLDPC_MAX_LANES], s_it[SCLDPC_MAX_LANES], s_ck[SCLDPC_MAX_LANES];
    if (threadIdx.x == 0) {
        p.cmp_cnt[g] = 0;
        int go = ld_cg(p.alive + g) != 0 && p.next_frame[g] >= p.frames_per_graph && p.gshift[g] > 0;
        int r = 0;
        for (int w = 0; w < W; w++) {
            s_act[w] = p.active[g * W + w];
            if (p.arm_mask[g * W + w] | p.done_mask[g * W + w]) go = 0;
            s_rank[w] = r;
            r += __popcll(s_act[w]);
        }
        s_rank[W] = r;
        if (go && (r < 1 || r > (64 << p.gshift[g]))) go = 0;    // worth it when the live frames fit into half the chunks in use
        s_go = go;
    }
    __syncthreads();
    if (!s_go) return;
    const int A = s_rank[W];
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_act[w] >> b) & 1ull) {
            const int i = s_rank[w] + __popcll(s_act[w] & ((1ull << b) - 1ull));
            p.cmp_src[g * p.lanes + i] = l;
            s_fr[i] = p.lane_frame[g * p.lanes + l];
            s_it[i] = p.lane_iter[g * p.lanes + l];
            if (p.stream_mode == SM_CKPT) s_ck[i] = p.lane_ck[g * p.lanes + l];
        }
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        p.lane_frame[g * p.lanes + l] = l < A ? s_fr[l] : -1;
        p.lane_iter[g * p.lanes + l] = l < A ? s_it[l] : 0;
        if (p.stream_mode == SM_CKPT) p.lane_ck[g * p.lanes + l] = l < A ? s_ck[l] : 0;
    }
    for (int w = threadIdx.x; w < W; w += blockDim.x)
        p.active[g * W + w] = A >= 64 * (w + 1) ? ~0ull : (A <= 64 * w ? 0ull : ((1ull << (A - 64 * w)) - 1ull));
    if (threadIdx.x == 0) {
        int s = 0;
        while ((128 << s) < A) s++;
        p.gshift[g] = s;
        p.cmp_cnt[g] = A;
        p.swept[2 * g] += 1;                                    // scldpc_bp_sweep_stats on a stream workspace: compactions, lanes moved
        p.swept[2 * g + 1] += A;
    }
}

#define CMP_ROWS 64
__global__ void __launch_bounds__(256) ns_compact_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y);
    const int A = ld_cg(p.cmp_cnt + g);
    if (A == 0) return;
    __shared__ unsigned short s_src[SCLDPC_MAX_LANES];
    __shared__ u128 s_in[CMP_ROWS * SCLDPC_MAX_WORDS / 2], s_out[CMP_ROWS * SCLDPC_MAX_WORDS / 2];
    const int ch = p.chunks, RWORDS = 2 * p.W, AW = (A + 31) >> 5;
    for (int i = threadIdx.x; i < A; i += blockDim.x) s_src[i] = (unsigned short)p.cmp_src[g * p.lanes + i];
    const unsigned *in32 = reinterpret_cast<const unsigned *>(s_in);
    unsigned *out32 = reinterpret_cast<unsigned *>(s_out);
    // tiles of the two planes' rows, then (streams with an unscanned head) of the cn_dis rows, which are per-lane decoder state too
    const int t_planes = (p.n + CMP_ROWS - 1) / CMP_ROWS;
    const int t_all = t_planes + (p.stream_mode == SM_HEAD ? (p.cn_dis_lim + CMP_ROWS - 1) / CMP_ROWS : 0);
    for (int t = blockIdx.x; t < t_all; t += gridDim.x) {
        const bool dis = t >= t_planes;
        const int row0 = (dis ? t - t_planes : t) * CMP_ROWS;
        const int rows = min(CMP_ROWS, (dis ? p.cn_dis_lim : p.n) - row0);
        u128 *__restrict__ x = dis ? p.cn_dis + (size_t)g * p.cn_dis_lim * ch : p.x + (size_t)g * p.n * ch;
        u128 *__restrict__ xb = dis ? nullptr : p.xb + (size_t)g * p.n * ch;
        __syncthreads();
        for (int i = threadIdx.x; i < rows * ch; i += blockDim.x) {
            s_in[i] = x[(size_t)row0 * ch + i];
            s_out[i] = zero128();
        }
        __syncthreads();
        for (int item = threadIdx.x; item < rows * AW; item += blockDim.x) {
            const int r = item / AW, q = item - r * AW;
            const unsigned *src = in32 + r * RWORDS;
            unsigned o = 0;
            const int nbits = min(32, A - 32 * q);
            for (int b = 0; b < nbits; b++) {
                const int l = s_src[32 * q + b];
                o |= ((src[l >> 5] >> (l & 31)) & 1u) << b;
            }
            out32[r * RWORDS + q] = o;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < rows * ch; i += blockDim.x) {
            const u128 v = s_out[i];
            if (neq(v, s_in[i])) {
                x[(size_t)row0 * ch + i] = v;
                if (xb) xb[(size_t)row0 * ch + i] = v;
            }
        }
    }
}

// x-plane row offsets of the CN edges (once per stream call)
__global__ void ns_cn_row_kernel(BpParams p)
{
    const int g = blockIdx.y;
    const size_t items = (size_t)p.nk * p.dc;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * items;
    int32_t *cn_row = p.cn_row + (size_t)g * items;
    // absent edges read the all-zero row that follows the last graph's plane
    const unsigned zero_row = (unsigned)(((size_t)(p.G - g) * p.n) << p.chunk_shift);
    if (blockIdx.x == 0 && threadIdx.x == 0) { p.gshift[g] = p.chunk_shift; p.cmp_cnt[g] = 0; }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (size_t)gridDim.x * blockDim.x) {
        const int e = cn_edge[i];
        cn_row[i] = (e != p.E) ? (int32_t)((unsigned)(e / p.dv) << p.chunk_shift) : (int32_t)zero_row;
    }
}

// ------------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------------
// every graph gets enough blocks to fill the machine on its own (blocks of finished graphs return at once); the same
// geometry for every launch of a stream call, because a warp replays the region it wrote itself
template <int DV, int DC>
static dim3 node_grid(const BpParams &p)
{
    const int block = 32 * NS_WARPS;
    static int res = 0;
    if (!res) {
        res = resident_blocks(ns_iter_kernel<DV, DC, SM_PLAIN>, block);
        if (res > NS_MAX_BLOCKS) res = NS_MAX_BLOCKS;
    }
    long long need = (((long long)p.cn_pos_lim * p.cns_pos << p.chunk_shift) + block - 1) / block;
    long long gx = need < res ? need : res;
    return dim3((unsigned)(gx < 1 ? 1 : gx), graphs_in_grid(p), 1);
}

template <int DV, int DC>
static void launch_node_iteration(const BpParams &p, bool after_harvest, cudaStream_t st)
{
    const dim3 block(32 * NS_WARPS), grid = node_grid<DV, DC>(p);
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += 1;
    // the first launch after a harvest follows ordinary kernels: full serialisation there
    const bool pdl = !after_harvest && !sample;
    switch (p.stream_mode) {
    case SM_CAPPED: launch_pdl(ns_iter_kernel<DV, DC, SM_CAPPED>, grid, block, st, pdl, p); break;
    case SM_CKPT: launch_pdl(ns_iter_kernel<DV, DC, SM_CKPT>, grid, block, st, pdl, p); break;
    case SM_HEAD:
        if (p.cn_dis_lim > 0) { launch_pdl(ns_iter_kernel<DV, DC, SM_HEAD>, grid, block, st, pdl, p); break; }
        [[fallthrough]];                                        // an empty head (is_bounded = True) leaves plain BP
    case SM_PLAIN: launch_pdl(ns_iter_kernel<DV, DC, SM_PLAIN>, grid, block, st, pdl, p); break;
    }
    if (sample) {
        cudaEventRecord(ev[1], st);
        cudaEventRecord(ev[2], st);                             // one kernel per iteration: the second interval is empty
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

// one iteration of every graph's frame stream; after_harvest: the launch follows the harvest kernels
int bp_launch_node_iteration(int dv, int dc, const BpParams &p, bool after_harvest, cudaStream_t st)
{
#define CALL_NI(A, B) launch_node_iteration<A, B>(p, after_harvest, st)
    SCLDPC_DISPATCH(dv, dc, CALL_NI);
#undef CALL_NI
    return 0;
}

// p.iter = the iteration that runs next; both planes equal and all lists empty afterwards
int bp_launch_node_settle(int dv, int dc, const BpParams &p, cudaStream_t st)
{
    dim3 grid;
#define CALL_NG(A, B) grid = node_grid<A, B>(p)
    SCLDPC_DISPATCH(dv, dc, CALL_NG);
#undef CALL_NG
    g_prof.launches += 2;
    ns_settle_kernel<<<grid, 32 * NS_WARPS, 0, st>>>(p);
    ns_settle_done_kernel<<<graphs_in_grid(p), 256, 0, st>>>(p);
    return 0;
}

void bp_launch_node_arm(const BpParams &p, cudaStream_t st)
{
    static int res = 0;
    if (!res) res = resident_blocks(ns_arm_kernel, 256);
    long long need = ((long long)p.n + ARM_ROWS - 1) / ARM_ROWS;
    long long gx = need < res ? need : res;
    g_prof.launches += 1;
    ns_arm_kernel<<<dim3((unsigned)(gx < 1 ? 1 : gx), graphs_in_grid(p)), 256, 0, st>>>(p);
}

// after the harvest and the arming: graphs in the tail of their stream move their live frames into the lowest lanes
void bp_launch_node_compact(const BpParams &p, cudaStream_t st)
{
    g_prof.launches += 2;
    ns_compact_plan_kernel<<<graphs_in_grid(p), 256, 0, st>>>(p);
    ns_compact_kernel<<<dim3(592, graphs_in_grid(p)), 256, 0, st>>>(p);
}

// list of the graphs still decoding after this harvest (ascending), for the grids of the launches the host enqueues once it has
// seen this harvest's counters
__global__ void ns_alive_list_kernel(BpParams p, int parity)
{
    int *list = p.glist2 + (size_t)parity * p.G, n = 0;                 // one warp: ballot + prefix, 32 graphs per trip
    const int lane = threadIdx.x & 31;
    for (int g0 = 0; g0 < p.G; g0 += 32) {
        const bool a = g0 + lane < p.G && p.alive[g0 + lane] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, a);
        if (a) list[n + __popc(m & ((1u << lane) - 1u))] = g0 + lane;
        n += __popc(m);
    }
    if (lane == 0) p.alive_total[6 + parity] = n;
}
void bp_launch_node_alive_list(const BpParams &p, int parity, cudaStream_t st)
{
    g_prof.launches += 1;
    ns_alive_list_kernel<<<1, 32, 0, st>>>(p, parity);
}

void bp_launch_node_tables(const BpParams &p, cudaStream_t st)
{
    g_prof.launches += 1;
    ns_cn_row_kernel<<<dim3(296, (unsigned)p.G), 256, 0, st>>>(p);
}

}  // namespace scldpc
