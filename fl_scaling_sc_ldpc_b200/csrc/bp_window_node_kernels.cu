// bp_window_node_kernels.cu -- window decoder (decodeBP_SW, BP_SW.c:628-912 / BP_FULL.c:627-897) and synchronous full BP
// without a trajectory in node-state form, ONE launch per flooding iteration (sm_100a).
//
// Schedule of the reference: per window the CN sweep covers CN positions [posW, posW+W) and the VN sweep the VN window
// (square: the same positions; classical: dv-1 more to the left); a VN outside the VN window keeps its outgoing messages,
// i.e. it looks to the CNs as it did when it was last swept.  Every VN a swept CN can resolve lies in the VN window or to
// its left, and a VN to the left of the window is never swept again (windows only move right) -- so what such a VN is told
// can never be seen by anybody.  The node state is therefore one bit per VN and frame, "erased as the CNs see it", which
// changes only for VNs of the VN window; resolutions that point to the left of it are dropped.
//
// As in bp_node_kernels.cu two equal planes alternate as read / write plane: the sweep reads one (flooding: every CN sees
// the state after the previous iteration), clears resolved bits in the other with red.and and logs (word, bit) per
// resolution in a per-warp region; the same warp of the next launch replays its region on that launch's write plane.
// Round 1 copied the pending plane over the visible one for the whole VN window after every CN sweep (a second launch that
// streamed 2 x 17 MB per graph at W = 10, 40 % of an iteration).
//
// Stopping per window (BP_SW.c:791-839): cap, NumErasuresTerm == NumErasuresPrecTerm (nothing resolved in the VN window;
// the first iteration compares with n, so it can only stall when the window holds all n VNs), NumErasuresTerm == 0.  The
// last one is detected one iteration late as "nothing resolved" and taken off again by the end-of-window kernel, which
// is the only pass over the VN window (once per window instead of once per iteration).  Frames that stopped keep their
// bits (FREEZE): resolutions are masked with the frames still iterating.
#include "common.cuh"

namespace scldpc {

// TRAJ (synchronous full BP with trajectory rows, BP_TRAJ.c:901-1151): the rows need, per frame and iteration, the degree-one
// counter, the newly resolved VNs and the first erased position.
//  * deg_1_iter (BP_TRAJ.c:935-979): a CN counts the first time one of its outgoing messages is "known" (latch), and only if
//    exactly one is.  With u erased neighbours in the read plane: no outgoing message is known for u >= 2, exactly one for
//    u = 1, all of them for u = 0 -- so the CN latches when u <= 1 and counts iff u = 1, or u = 0 and it has a single edge.
//    (The extrinsic messages can differ from the a-posteriori state only for a VN that this CN itself resolved, and then
//    the CN has latched before.)  Counted per lane without atomics (LaneCounter, common.cuh).
//  * dVNs, first erased position, NumErasures: per (position, lane) counters of erased VNs, initialised from the channel and
//    decremented by the thread that actually clears a bit (atom.and returns the old word, so a VN resolved by two CNs in the
//    same iteration is counted once).  The last block sums them per lane: NumErasures is exact, so frames stop in the
//    iteration the reference stops in (no late "finished" stop, no end-of-window correction).
template <int DV, int DC, bool HEAD, bool TRAJ>
__global__ void __launch_bounds__(32 * NS_WARPS, TRAJ ? 3 : 4) bpw_iter_kernel(BpParams p)
{
    static_assert(DC <= 16, "neighbour index is encoded in four bit planes");
    pdl_wait_then_release();
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ u64 s_new[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    __shared__ int s_cnt[TRAJ ? SCLDPC_MAX_LANES : 1];
    __shared__ u128 s_planes[TRAJ ? LC_PLANES * 32 * NS_WARPS : 1];
    if (threadIdx.x < SCLDPC_MAX_WORDS) s_new[threadIdx.x] = 0;
    if (TRAJ)
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
    LaneCounter lc;
    if (TRAJ) lc.clear();
    __syncthreads();
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int par = p.iter & 1;
    const size_t plane = (size_t)g * p.n * ch;
    const u128 *__restrict__ rd = (par ? p.xb : p.x) + plane;
    u128 *__restrict__ wr = (par ? p.x : p.xb) + plane;
    unsigned *__restrict__ wr32 = reinterpret_cast<unsigned *>(wr);
    const int RW = p.nl_rw;
    const int rid = blockIdx.x * NS_WARPS + warp;

    // ---- the write plane catches up with the previous iteration (nothing to do in a window's first iteration) ----
    if (ld_cg(p.nl_ovf + g * 2 + (par ^ 1))) ns_catch_up(rd, wr, p.v0 << p.chunk_shift, p.v1 << p.chunk_shift);
    else ns_replay_region(p, g, par ^ 1, wr32, rid, false);

    // ---- check-node sweep over [c0, c1) ----
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const bool lane_work = nz(act);                             // a thread keeps its chunk
    const u128 *__restrict__ rdk = rd + k;
    const int32_t *__restrict__ cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    uint2 *__restrict__ reg = p.nl_list + ((size_t)(g * 2 + par) * RW + rid) * p.nl_stride;
    const int items = (p.c1 - p.c0) << p.chunk_shift;
    const int stride = gridDim.x * blockDim.x;
    const int E = p.E;
    const unsigned lo = (unsigned)p.v0, span = (unsigned)(p.v1 - p.v0);
    int wcount = 0;                                             // entries this warp has logged (warp-uniform)
    unsigned acc_new[4] = {0u, 0u, 0u, 0u};                     // frames that resolved a VN of the VN window
    int trip = 0;                                               // block-uniform trip count (the counter flush is a block-wide step)
    for (int base = blockIdx.x * blockDim.x; base < items; base += stride, trip++) {
        const int idx = base + threadIdx.x;
        u128 res = zero128(), b0 = zero128(), b1 = zero128(), b2 = zero128(), b3 = zero128();
        const int c = p.c0 + (idx >> p.chunk_shift);
        const int32_t *row = cn_edge + (size_t)c * DC;
        if (lane_work && idx < items) {
            int e[DC];
            load_row<DC>(row, e);
            u128 in[DC];
#pragma unroll
            for (int j = 0; j < DC; j++) in[j] = (e[j] != E) ? ld_stream(rdk + (unsigned)((e[j] / DV) << p.chunk_shift)) : zero128();
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
            res = one & ~tw & act;                              // exactly one erased neighbour, frame still iterating
            if (TRAJ) {
                int deg = 0;
#pragma unroll
                for (int j = 0; j < DC; j++) deg += (e[j] != E);
                if (deg > 0) {
                    u128 *lp = p.latch + ((size_t)g * p.nk + c) * ch + k;
                    const u128 lat = *lp;
                    const u128 nl = lat | (~tw & act);
                    if (neq(nl, lat)) *lp = nl;
                    lc.add((deg == 1 ? ~tw : (one & ~tw)) & ~lat & act);
                }
            }
            if (HEAD && c < p.cn_dis_lim) {
                // Unscanned head of simulate_sc_ldpc (is_bounded = False): a slot below the scan start is only decoded when a
                // removal leaves it with one user (PD.py:308-311), so a CN that starts with exactly one erased neighbour never
                // resolves it (same plane as bp_cn_wave_kernel<.,.,HEAD>)
                u128 *dp = p.cn_dis + ((size_t)g * p.cn_dis_lim + c) * ch + k;
                u128 dis;
                if (p.first_iter) { dis = one & ~tw; *dp = dis; }
                else dis = *dp;
                res &= ~dis;
            }
        }
        if (TRAJ && (trip % 31) == 30) lane_counter_flush(lc, s_planes, s_cnt, ch);
        if (__ballot_sync(0xffffffffu, nz(res)) == 0u) continue;
        const int cnt = __popcll(res.x) + __popcll(res.y);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        int slot = wcount + incl - cnt;
        wcount += __shfl_sync(0xffffffffu, incl, 31);
        if (cnt) {
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
                    const unsigned v = (unsigned)__ldg(row + j) / DV;                          // L1 hit
                    uint2 entry = make_uint2(0u, 0u);
                    if (v - lo < span) {                         // a VN of the VN window: the only ones anybody will look at again
                        const unsigned widx = 4u * ((v << p.chunk_shift) + (unsigned)k) + (unsigned)q;
                        if (!TRAJ) red_and(wr32 + widx, ~(1u << b));
                        else if (slot >= p.nl_cap) {
                            // (region full: clear and count in place; otherwise after the sweep, see below)
                            const unsigned old = atomicAnd(wr32 + widx, ~(1u << b));
                            if ((old >> b) & 1u)
                                atomicSub(p.pos_pairs + ((size_t)g * p.L + v / (unsigned)p.vns_pos) * p.lanes + k * 128 + q * 32 + b, 1);
                        }
                        entry = make_uint2(widx, 1u << b);
                        acc_new[q] |= 1u << b;
                    }
                    if (slot < p.nl_cap) st_cg_u2(reg + slot, entry);
                    slot++;
                }
            }
        }
    }
    if (lane == 0) {
        p.nl_cnt[(size_t)(g * 2 + par) * RW + rid] = wcount < p.nl_cap ? wcount : p.nl_cap;
        if (wcount > p.nl_cap) p.nl_ovf[g * 2 + par] = 1;
    }
    if (TRAJ) {
        // Clearing + counting of this iteration's resolutions, from the warp's own list: the thread whose atom.and finds the
        // bit still set takes the VN off its position's count (a VN resolved by two CNs in one iteration is counted once).
        // Done here rather than in the sweep so that eight atomics with a return value are in flight per thread -- in the
        // sweep every trip waited for its own (161 -> see DESIGN.md section 5).
        __syncwarp();
        const int cnt = wcount < p.nl_cap ? wcount : p.nl_cap;
        constexpr int U = 8;
        for (int i0 = lane; i0 < cnt; i0 += 32 * U) {
            uint2 e[U];
            unsigned old[U];
#pragma unroll
            for (int u = 0; u < U; u++) e[u] = (i0 + 32 * u < cnt) ? ld_cg_u2(reg + i0 + 32 * u) : make_uint2(0u, 0u);
#pragma unroll
            for (int u = 0; u < U; u++) old[u] = e[u].y ? atomicAnd(wr32 + e[u].x, ~e[u].y) : 0u;
#pragma unroll
            for (int u = 0; u < U; u++)
                if (old[u] & e[u].y) {
                    const unsigned row = e[u].x >> (2 + p.chunk_shift), kk = (e[u].x >> 2) & (unsigned)(ch - 1), qq = e[u].x & 3u;
                    atomicSub(p.pos_pairs + ((size_t)g * p.L + row / (unsigned)p.vns_pos) * p.lanes + kk * 128 + qq * 32 + (__ffs((int)e[u].y) - 1), 1);
                }
        }
        lane_counter_flush(lc, s_planes, s_cnt, ch);
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(p.cnt_deg1 + ((size_t)g * SCLDPC_CNT_SLOTS + (blockIdx.x % SCLDPC_CNT_SLOTS)) * p.lanes + i, s_cnt[i]);
    }
    u128 an = make_u128((u64)acc_new[0] | ((u64)acc_new[1] << 32), (u64)acc_new[2] | ((u64)acc_new[3] << 32));
    an = warp_or_same_chunk(an, ch);
    if (lane < ch) {
        if (an.x) atomicOr(&s_new[2 * k], an.x);
        if (an.y) atomicOr(&s_new[2 * k + 1], an.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_new[w] & ~ld_cg(p.any_new + g * p.W + w)) atomicOr(p.any_new + g * p.W + w, s_new[w]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- end of the iteration for graph g (bp_retire_lanes without the "no erasure left" test, see the file header) ----
    __shared__ u64 s_stop[SCLDPC_MAX_WORDS];
    __shared__ u64 s_er[SCLDPC_MAX_WORDS], s_prog[SCLDPC_MAX_WORDS];
    __shared__ int s_alive;
    if (threadIdx.x == 0) s_alive = 0;
    if (threadIdx.x < SCLDPC_MAX_WORDS) { s_er[threadIdx.x] = 0; s_prog[threadIdx.x] = 0; }
    __syncthreads();
    if (TRAJ) {
        // per lane: NumErasures, the row of this iteration (BP_TRAJ.c:988,1051), "an erased VN is left", "a VN was resolved"
        for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
            int cur = 0, first = p.L;                                   // first_erased = n => prints L (BP_TRAJ.c:1017,1051)
            for (int q = 0; q < p.L; q++) {
                const int v = ld_cg(p.pos_pairs + ((size_t)g * p.L + q) * p.lanes + l);
                if (v > 0 && first == p.L) first = q;
                cur += v;
            }
            int d1 = 0;
            for (int sl = 0; sl < SCLDPC_CNT_SLOTS; sl++) {
                const size_t o = ((size_t)g * SCLDPC_CNT_SLOTS + sl) * p.lanes + l;
                d1 += ld_cg(p.cnt_deg1 + o);
                p.cnt_deg1[o] = 0;
            }
            const int prev = p.cnt_dvn[(size_t)g * SCLDPC_CNT_SLOTS * p.lanes + l];      // NumErasuresPrec
            const int w = l >> 6, b = l & 63;
            if ((p.active[g * p.W + w] >> b) & 1ull) {
                if (p.row >= 0 && p.row < p.max_rows) {
                    int *r = p.rows + (((size_t)g * p.max_rows + p.row) * p.lanes + l) * 3;
                    r[0] = d1; r[1] = prev - cur; r[2] = first;
                }
                p.cnt_dvn[(size_t)g * SCLDPC_CNT_SLOTS * p.lanes + l] = cur;
                if (cur > 0) atomicOr(reinterpret_cast<unsigned long long *>(&s_er[w]), 1ull << b);
                if (prev != cur) atomicOr(reinterpret_cast<unsigned long long *>(&s_prog[w]), 1ull << b);
            }
        }
        __syncthreads();
    }
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        const u64 a = p.active[g * p.W + w];
        u64 nw = ld_cg(p.any_new + g * p.W + w);
        u64 stop = 0;
        if (TRAJ) stop = a & (~s_er[w] | ~s_prog[w]);                   // NumErasures == 0 || == NumErasuresPrec (exact counts)
        else if (!p.first_iter) stop = a & ~nw;                         // NumErasuresTerm == NumErasuresPrecTerm
        else if (p.stall_at_first) stop = a & ~(nw | p.win_known[g * p.W + w]);   // ... == n: nothing resolved and nothing known
        if (!TRAJ) p.noprog[g * p.W + w] |= stop;
        if (p.iter + 1 >= p.max_it) stop = a;                           // while (iter < NumIt)
        s_stop[w] = stop;
        const u64 left = a & ~stop;
        p.active[g * p.W + w] = left;
        p.any_new[g * p.W + w] = 0;
        if (left) s_alive = 1;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_stop[w] >> b) & 1ull) {
            p.iters[g * p.lanes + l] += p.iter + 1;
            p.work[g * p.lanes + l] += (long long)(p.iter + 1) * p.win_edges;
        }
    }
    if (threadIdx.x == 0) {
        p.nl_ovf[g * 2 + (par ^ 1)] = 0;                        // consumed by every block of this launch
        p.nl_last[g] = p.iter;
        p.ticket[g] = 0;
        if (!s_alive) { p.alive[g] = 0; atomicSub(p.alive_total, 1); }
    }
}

// End of a window (same grid as the iteration kernel): the plane the last executed iteration read catches up (both planes
// equal, lists empty), and the one pass over the VN window finds the frames that stopped on "nothing resolved" with no
// erased VN left in the window -- the reference had stopped them one iteration earlier (NumErasuresTerm == 0).
__global__ void __launch_bounds__(32 * NS_WARPS) bpw_window_end_kernel(BpParams p)
{
    const int g = blockIdx.y;
    const int last = ld_cg(p.nl_last + g);
    if (last < 0) return;                                       // no iteration ran for this graph in this window
    __shared__ u64 s_er[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (threadIdx.x < SCLDPC_MAX_WORDS) s_er[threadIdx.x] = 0;
    __syncthreads();
    const int ch = p.chunks, k = threadIdx.x & (ch - 1);
    const int par = last & 1;                                   // the last iteration read plane `par`, wrote the other and logged list `par`
    const size_t plane = (size_t)g * p.n * ch;
    u128 *stale = (par ? p.xb : p.x) + plane;
    const u128 *fresh = (par ? p.x : p.xb) + plane;
    if (ld_cg(p.nl_ovf + g * 2 + par)) {
        ns_catch_up(fresh, stale, p.v0 << p.chunk_shift, p.v1 << p.chunk_shift);
        if ((threadIdx.x & 31) == 0) p.nl_cnt[(size_t)(g * 2 + par) * p.nl_rw + blockIdx.x * NS_WARPS + (threadIdx.x >> 5)] = 0;
    } else ns_replay_region(p, g, par, reinterpret_cast<unsigned *>(stale), blockIdx.x * NS_WARPS + (threadIdx.x >> 5), true);
    // erased VNs left in the VN window, for the frames that stopped on "nothing resolved"
    const u128 np = reinterpret_cast<const u128 *>(p.noprog)[g * ch + k];
    u128 er = zero128();
    if (nz(np)) {
        const int i0 = p.v0 << p.chunk_shift, i1 = p.v1 << p.chunk_shift;
        for (int i = i0 + blockIdx.x * blockDim.x + threadIdx.x; i < i1; i += gridDim.x * blockDim.x) er |= ld_cg128(fresh + i);
        er &= np;
    }
    er = warp_or_same_chunk(er, ch);
    if ((threadIdx.x & 31) < ch) {
        if (er.x) atomicOr(&s_er[2 * k], er.x);
        if (er.y) atomicOr(&s_er[2 * k + 1], er.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_er[w] & ~ld_cg(p.any_er + g * p.W + w)) atomicOr(p.any_er + g * p.W + w, s_er[w]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        const u64 early = p.noprog[g * p.W + w] & ~ld_cg(p.any_er + g * p.W + w);
        if ((early >> b) & 1ull) {
            p.iters[g * p.lanes + l] -= 1;
            p.work[g * p.lanes + l] -= p.win_edges;
        }
    }
    __syncthreads();
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) { p.noprog[g * p.W + w] = 0; p.any_er[g * p.W + w] = 0; }
    if (threadIdx.x == 0) {
        p.nl_ovf[g * 2 + par] = 0;
        p.nl_last[g] = -1;
        p.ticket[g] = 0;
    }
}

// ------------------------------------------------------------------------------------------------------------
// Copy variant (round 1), kept for windows that are short against the chain.  Inside a window the wave is everywhere: a third
// to a half of the window's rows change per iteration, so logging and replaying every resolution costs more than copying the
// window (measured on B200, L = 100, M = 10000, 4 x 1024 frames: lists 87 / 72 / 63 k frames/s at W = 3 / 5 / 10 against 112 /
// 100 / 69 k with the copy).  Here x is what the CNs see and xb what every VN has been told; the CN sweep clears bits in xb, a
// second launch copies xb over x on the VN window and evaluates the reference's stop rules exactly (no late stop).
// The list variant above serves sweeps over (most of) the chain: synchronous full BP, long windows.
// ------------------------------------------------------------------------------------------------------------
template <int DV, int DC, bool HEAD>
__global__ void __launch_bounds__(256, 4) bpw_cn_copy_kernel(BpParams p)
{
    static_assert(DC <= 16, "neighbour index is encoded in four bit planes");
    pdl_wait_then_release();
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    if (!nz(act)) return;                                       // a thread keeps its chunk
    const u128 *__restrict__ xk = p.x + (size_t)g * p.n * ch + k;
    unsigned *__restrict__ xbk = reinterpret_cast<unsigned *>(p.xb + (size_t)g * p.n * ch + k);
    const int32_t *__restrict__ cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const int items = (p.c1 - p.c0) << p.chunk_shift;
    const int stride = gridDim.x * blockDim.x;
    const int E = p.E;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += stride) {
        const int32_t *row = cn_edge + (size_t)(p.c0 + (idx >> p.chunk_shift)) * DC;
        int e[DC];
        load_row<DC>(row, e);
        u128 in[DC];
#pragma unroll
        for (int j = 0; j < DC; j++) in[j] = (e[j] != E) ? ld_stream(xk + (unsigned)((e[j] / DV) << p.chunk_shift)) : zero128();
        u128 one = zero128(), tw = zero128(), b0 = zero128(), b1 = zero128(), b2 = zero128(), b3 = zero128();
#pragma unroll
        for (int j = 0; j < DC; j++) {
            tw |= one & in[j];
            one |= in[j];
            if (j & 1) b0 |= in[j];
            if (j & 2) b1 |= in[j];
            if (j & 4) b2 |= in[j];
            if (j & 8) b3 |= in[j];
        }
        u128 res = one & ~tw & act;                             // exactly one erased neighbour, frame still iterating
        if (HEAD && p.c0 + (idx >> p.chunk_shift) < p.cn_dis_lim) {
            // Unscanned head of simulate_sc_ldpc (is_bounded = False): a slot below the scan start is only decoded when a
            // removal leaves it with one user (PD.py:308-311), so a CN that starts with exactly one erased neighbour never
            // resolves it (same plane as bp_cn_wave_kernel<.,.,HEAD>)
            u128 *dp = p.cn_dis + ((size_t)g * p.cn_dis_lim + p.c0 + (idx >> p.chunk_shift)) * ch + k;
            u128 dis;
            if (p.first_iter) { dis = one & ~tw; *dp = dis; }
            else dis = *dp;
            res &= ~dis;
        }
        if (nz(res)) {
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
                    const unsigned o = (unsigned)((__ldg(row + j) / DV) << p.chunk_shift);
                    red_and(xbk + 4 * (size_t)o + q, ~(1u << b));
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256, 4) bpw_vn_copy_kernel(BpParams p)
{
    pdl_wait_then_release();
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ u64 s_new[SCLDPC_MAX_WORDS], s_er[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (threadIdx.x < SCLDPC_MAX_WORDS) { s_new[threadIdx.x] = 0; s_er[threadIdx.x] = 0; }
    __syncthreads();
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    u128 acc_new = zero128(), acc_er = zero128();
    u128 *__restrict__ x = p.x + ((size_t)g * p.n + p.v0) * ch;
    const u128 *__restrict__ xb = p.xb + ((size_t)g * p.n + p.v0) * ch;
    const int items = (p.v1 - p.v0) << p.chunk_shift;
    const int stride = gridDim.x * blockDim.x;
    constexpr int U = 4;                                        // rows in flight per thread: a plain stream, latency-bound otherwise
    if (nz(act))
        for (int base = blockIdx.x * blockDim.x * U + threadIdx.x; base < items; base += stride * U) {
            u128 xos[U], xbs[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int idx = base + u * (int)blockDim.x;
                xos[u] = zero128(); xbs[u] = zero128();
                if (idx < items) { xos[u] = x[idx]; xbs[u] = ld_cg128(xb + idx); }   // the CN sweep wrote xb with atomics (L2)
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int idx = base + u * (int)blockDim.x;
                if (idx >= items) break;
                const u128 xo = xos[u];
                const u128 xn = sel(act, xbs[u], xo);
                if (neq(xn, xo)) x[idx] = xn;
                // a window's first iteration compares with NumErasuresPrecTerm = n: "progress" = some VN of the range is known
                acc_new |= (p.first_iter ? ~xn : (xo & ~xn)) & act;
                acc_er |= xn & act;
            }
        }
    acc_new = warp_or_same_chunk(acc_new, ch);
    acc_er = warp_or_same_chunk(acc_er, ch);
    if ((threadIdx.x & 31) < ch) {
        if (acc_new.x) atomicOr(&s_new[2 * k], acc_new.x);
        if (acc_new.y) atomicOr(&s_new[2 * k + 1], acc_new.y);
        if (acc_er.x) atomicOr(&s_er[2 * k], acc_er.x);
        if (acc_er.y) atomicOr(&s_er[2 * k + 1], acc_er.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_new[w] & ~ld_cg(p.any_new + g * p.W + w)) atomicOr(p.any_new + g * p.W + w, s_new[w]);
        if (s_er[w] & ~ld_cg(p.any_er + g * p.W + w)) atomicOr(p.any_er + g * p.W + w, s_er[w]);
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        bp_retire_lanes<false>(p, g);
    }
}

// x = xb = channel erasures (Lji = channel value on every edge, Lij = 1: BP_SW.c:650-659); win_known = frames in which the
// channel left some VN known (the first iteration of a window that holds all n VNs compares with NumErasuresPrec = n)
__global__ void bpw_node_init_kernel(BpParams p)
{
    const size_t items = (size_t)p.G * p.n * p.chunks;
    const u128 *chan = reinterpret_cast<const u128 *>(p.chan);
    const int ch = p.chunks;
    u128 known = zero128();
    int g_cur = -1;
    auto flush = [&]() {
        if (g_cur >= 0 && nz(known)) {
            const int k = threadIdx.x & (ch - 1);
            if (known.x) atomicOr(reinterpret_cast<unsigned long long *>(p.win_known + g_cur * p.W + 2 * k), known.x);
            if (known.y) atomicOr(reinterpret_cast<unsigned long long *>(p.win_known + g_cur * p.W + 2 * k + 1), known.y);
        }
        known = zero128();
    };
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(i / ((size_t)p.n * ch));
        if (g != g_cur) { flush(); g_cur = g; }
        const u128 c = chan[i];
        p.x[i] = c;
        p.xb[i] = c;
        known |= ~c;
    }
    flush();
}

// trajectory mode: NumErasuresPrec = n for every frame (BP_TRAJ.c:910); the per-position counts come from bp_pos_count_kernel
__global__ void bpw_traj_init_kernel(BpParams p)
{
    const int g = blockIdx.x;
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) p.cnt_dvn[(size_t)g * SCLDPC_CNT_SLOTS * p.lanes + l] = p.n;
}

__global__ void bpw_node_reset_kernel(BpParams p, int zero_known)
{
    const int RW = p.nl_rw;
    const int g = blockIdx.x;
    for (int i = threadIdx.x; i < 2 * RW; i += blockDim.x) p.nl_cnt[(size_t)g * 2 * RW + i] = 0;
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        p.noprog[g * p.W + w] = 0;
        p.win_known[g * p.W + w] = zero_known ? 0ull : ~0ull;
    }
    if (threadIdx.x == 0) { p.nl_ovf[2 * g] = 0; p.nl_ovf[2 * g + 1] = 0; p.nl_last[g] = -1; }
}

// ------------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------------
template <int DV, int DC>
static dim3 window_grid(const BpParams &p)
{
    const int block = 32 * NS_WARPS;
    static int res = 0;
    if (!res) {
        res = resident_blocks(bpw_iter_kernel<DV, DC, false, false>, block);
        if (res > NS_MAX_BLOCKS) res = NS_MAX_BLOCKS;
    }
    // the same geometry for every launch of a window (a warp replays the region it wrote itself): a function of the ranges only
    long long items = (long long)(p.c1 - p.c0) << p.chunk_shift;
    const long long vitems = (long long)(p.v1 - p.v0) << p.chunk_shift;
    if (vitems / 4 > items) items = vitems / 4;                  // the end-of-window pass over the VN window uses this grid too
    long long need = (items + block - 1) / block;
    long long gx = need < res ? need : res;
    return dim3((unsigned)(gx < 1 ? 1 : gx), (unsigned)p.G, 1);
}

template <int DV, int DC>
static void launch_window_copy_iteration(const BpParams &p, cudaStream_t st)
{
    const int block = 256;
    dim3 gc = sweep_grid((long long)(p.c1 - p.c0) << p.chunk_shift, p.G, block, SWEEP_BLOCKS_PER_SM);
    dim3 gv = sweep_grid((((long long)(p.v1 - p.v0) << p.chunk_shift) + 3) / 4, p.G, block, SWEEP_BLOCKS_PER_SM);   // four rows per thread and trip
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += (p.c1 > p.c0) ? 2 : 1;
    // programmatic dependent launches inside a window / a call; its first kernel follows ordinary ones
    const bool pdl = !sample;
    if (p.c1 > p.c0) {
        if (p.cn_dis_lim > 0) launch_pdl(bpw_cn_copy_kernel<DV, DC, true>, gc, dim3(block), st, pdl && !p.first_iter, p);
        else launch_pdl(bpw_cn_copy_kernel<DV, DC, false>, gc, dim3(block), st, pdl && !p.first_iter, p);
    }
    if (sample) cudaEventRecord(ev[1], st);
    launch_pdl(bpw_vn_copy_kernel, gv, dim3(block), st, pdl && (p.c1 > p.c0 || !p.first_iter), p);
    if (sample) {
        cudaEventRecord(ev[2], st);
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

template <int DV, int DC>
static void launch_window_node_iteration(const BpParams &p, cudaStream_t st)
{
    const dim3 block(32 * NS_WARPS), grid = window_grid<DV, DC>(p);
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += 1;
    // programmatic dependent launches inside a window; its first kernel follows ordinary ones
    const bool pdl = !sample && !p.first_iter;
    if (p.traj_node) launch_pdl(bpw_iter_kernel<DV, DC, false, true>, grid, block, st, pdl, p);
    else if (p.cn_dis_lim > 0) launch_pdl(bpw_iter_kernel<DV, DC, true, false>, grid, block, st, pdl, p);
    else launch_pdl(bpw_iter_kernel<DV, DC, false, false>, grid, block, st, pdl, p);
    if (sample) {
        cudaEventRecord(ev[1], st);
        cudaEventRecord(ev[2], st);                             // one kernel per iteration: the second interval is empty
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

int bp_launch_window_node_iteration(int dv, int dc, const BpParams &p, cudaStream_t st)
{
    if (!p.win_lists) {
#define CALL_WC(A, B) launch_window_copy_iteration<A, B>(p, st)
        SCLDPC_DISPATCH(dv, dc, CALL_WC);
#undef CALL_WC
        return 0;
    }
#define CALL_WI(A, B) launch_window_node_iteration<A, B>(p, st)
    SCLDPC_DISPATCH(dv, dc, CALL_WI);
#undef CALL_WI
    return 0;
}

// after the iterations of a window (or of a synchronous full-BP call): settle the planes, undo the late "finished" stops
int bp_launch_window_node_end(int dv, int dc, const BpParams &p, cudaStream_t st)
{
    if (!p.win_lists) return 0;                                  // the copy variant leaves nothing pending
    dim3 grid;
#define CALL_WG(A, B) grid = window_grid<A, B>(p)
    SCLDPC_DISPATCH(dv, dc, CALL_WG);
#undef CALL_WG
    g_prof.launches += 1;
    bpw_window_end_kernel<<<grid, 32 * NS_WARPS, 0, st>>>(p);
    return 0;
}

void bp_launch_window_node_traj_init(const BpParams &p, cudaStream_t st)
{
    g_prof.launches += 1;
    bpw_traj_init_kernel<<<p.G, 256, 0, st>>>(p);
}

// resume: the caller supplied both planes (scldpc_bp_window_range), only the list bookkeeping is reset
void bp_launch_window_node_init(const BpParams &p, cudaStream_t st, bool resume)
{
    g_prof.launches += resume ? 1 : 2;
    bpw_node_reset_kernel<<<p.G, 256, 0, st>>>(p, resume ? 0 : 1);
    if (!resume) bpw_node_init_kernel<<<num_sms() * 8, 256, 0, st>>>(p);
}

}  // namespace scldpc
