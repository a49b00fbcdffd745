// bp_wave_kernels.cu -- full flooding BP with wave tracking (sm_100a).
//
// Decoding an SC-LDPC code is a travelling wave: after a short transient only the ~10 positions around each wave
// front change, positions behind a front are resolved and positions ahead of it sit at a fixed point of the local
// rule.  The reference sweeps all L(+dv-1) positions in every iteration (BP_FULL.c:943,985,1009).  Here a sweep
// visits a position only if one of its inputs changed since it was last computed -- which leaves every message,
// every decision and every counter bit-identical, because a node whose inputs did not change recomputes its old
// outputs:
//   * a VN's outgoing messages are a function of its state (x, y): x = a-posteriori erasure, y = "some outgoing
//     message is an erasure" (incoming Lij only go 1->0, so the state walks 4 erased -> 3 erased -> <=2 erased and
//     the outgoing messages change exactly when (x, y) changes).  The VN sweep compares (x, y) with the stored
//     planes and stamps its position when any active frame changed;
//   * CN position p is swept in iteration t iff a VN position in [p-dv+1, p] was stamped in iteration t-1;
//   * VN position q is swept in iteration t iff a CN position in [q, q+dv-1] was swept in iteration t.
// The lists are rebuilt on the device by the last block of each VN sweep.  Messages of VNs that did not change
// are not written back.  Besides doing less work, the live region (a few tens of MB) stays resident in the 126 MB
// L2 across iterations, so most of its traffic never reaches HBM.
//
// Useful work is still accounted as the reference's: 2E edge updates per frame-iteration.
#include <climits>

#include "common.cuh"

namespace scldpc {

// ------------------------------------------------------------------------------------------------------------
__global__ void bp_wave_init_kernel(BpParams p)
{
    const int g = blockIdx.x;
    const int ncp = p.L + p.dv - 1;
    for (int i = threadIdx.x; i < ncp; i += blockDim.x) p.cn_list[g * ncp + i] = i;
    for (int i = threadIdx.x; i < p.L; i += blockDim.x) {
        p.vn_list[g * p.L + i] = i;
        p.vn_stamp[g * p.L + i] = -1;
    }
    for (int i = threadIdx.x; i < p.L * p.W; i += blockDim.x) p.pos_er_new[(size_t)g * p.L * p.W + i] = 0;
    if (threadIdx.x == 0) {
        p.n_list[2 * g] = p.cn_pos_lim;
        p.n_list[2 * g + 1] = p.L;
        p.swept[2 * g] = 0;
        p.swept[2 * g + 1] = 0;
    }
}

// ------------------------------------------------------------------------------------------------------------
// check-node sweep over the listed positions
// ------------------------------------------------------------------------------------------------------------
template <int DC, bool TRAJ, bool HEAD = false>
__global__ void __launch_bounds__(256, (TRAJ || HEAD) ? 3 : 5) bp_cn_wave_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y);
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ int s_cnt[TRAJ ? SCLDPC_MAX_LANES : 1];
    __shared__ u128 s_planes[TRAJ ? LC_PLANES * 256 : 1];
    if (TRAJ) {
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
        __syncthreads();
    }
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const u128 *__restrict__ v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
    u128 *__restrict__ c2v = p.c2v + (size_t)g * p.nk * DC * ch;
    const int32_t *__restrict__ cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const int *__restrict__ list = p.cn_list + g * (p.L + p.dv - 1);
    LaneCounter lc;
    if (TRAJ) lc.clear();

    const bool lane_work = nz(act);
    const int ipp = p.cns_pos << p.chunk_shift;                 // work items per position
    const int items = ld_cg(p.n_list + 2 * g) * ipp;
    const int stride = gridDim.x * blockDim.x;
    // In trajectory mode the trip count is block-uniform (the counter flush below is a block-wide step).
    int trip = 0;
    for (int base = blockIdx.x * blockDim.x; base < items; base += stride, trip++) {
        const int idx = base + threadIdx.x;
        if (lane_work && idx < items) {
            const int ent = idx / ipp, off = idx - ent * ipp;
            const int c = __ldg(list + ent) * p.cns_pos + (off >> p.chunk_shift);
            int e[DC];
            load_row<DC>(cn_edge + (size_t)c * DC, e);
            u128 in[DC];
#pragma unroll
            for (int j = 0; j < DC; j++) in[j] = ld_stream(v2c + (size_t)e[j] * ch + k);
            u128 out[DC];
            u128 acc = zero128();
#pragma unroll
            for (int j = 0; j < DC; j++) { out[j] = acc; acc |= in[j]; }
            acc = zero128();
#pragma unroll
            for (int j = DC - 1; j >= 0; j--) { out[j] |= acc; acc |= in[j]; }
            if (HEAD && c < p.cn_dis_lim) {
                // Unscanned head of simulate_sc_ldpc (is_bounded = False): a slot below the scan start is only decoded
                // when a removal leaves it with one user (subtract_interference, PD.py:308-311), so a CN that starts with
                // exactly one erased neighbour never resolves it: its outgoing messages stay erasures.
                u128 *dp = p.cn_dis + ((size_t)g * p.cn_dis_lim + c) * ch + k;
                u128 dis;
                if (p.first_iter) {
                    u128 one = zero128(), two = zero128();
#pragma unroll
                    for (int j = 0; j < DC; j++) { two |= one & in[j]; one |= in[j]; }
                    dis = one & ~two;
                    *dp = dis;
                } else dis = *dp;
#pragma unroll
                for (int j = 0; j < DC; j++) out[j] |= dis;
            }
            u128 *dst = c2v + ((size_t)c * DC) * ch + k;
#pragma unroll
            for (int j = 0; j < DC; j++) dst[(size_t)j * ch] = out[j];
            if (TRAJ) {
                // degree-one counter with latch (BP_FULL.c:935-979): num_out_resolved = #j with out[j] == 0
                u128 one = zero128(), two = zero128();
#pragma unroll
                for (int j = 0; j < DC; j++) {
                    if (e[j] != p.E) { u128 z = ~out[j]; two |= one & z; one |= z; }
                }
                u128 *lp = p.latch + ((size_t)g * p.nk + c) * ch + k;
                const u128 lat = *lp;
                const u128 nl = lat | (one & act);
                if (neq(nl, lat)) *lp = nl;
                lc.add(one & ~two & ~lat & act);
            }
        }
        if (TRAJ && (trip % 31) == 30) lane_counter_flush(lc, s_planes, s_cnt, ch);
    }
    if (TRAJ) {
        lane_counter_flush(lc, s_planes, s_cnt, ch);
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(p.cnt_deg1 + ((size_t)g * SCLDPC_CNT_SLOTS + (blockIdx.x % SCLDPC_CNT_SLOTS)) * p.lanes + i, s_cnt[i]);
    }
}

// ------------------------------------------------------------------------------------------------------------
// end of an iteration (last block of the VN sweep): retire frames, rebuild the position lists
// ------------------------------------------------------------------------------------------------------------
template <bool TRAJ>
__device__ void bp_wave_retire(const BpParams &p, int g)
{
    __shared__ u64 s_stop[SCLDPC_MAX_WORDS], s_act[SCLDPC_MAX_WORDS];
    __shared__ int s_alive;
    __shared__ unsigned char s_chg[1024 + 16], s_cn[1024 + 16];
    const int L = p.L, W = p.W, ncp = L + p.dv - 1;
    const int n_vn = p.n_list[2 * g + 1];
    if (threadIdx.x == 0) s_alive = 0;
    // positions swept in this iteration publish their "erased VN left" words
    for (int i = threadIdx.x; i < n_vn * W; i += blockDim.x) {
        const int pos = p.vn_list[g * L + i / W], w = i % W;
        const size_t o = ((size_t)g * L + pos) * W + w;
        p.pos_er[o] = ld_cg(p.pos_er_new + o);
        p.pos_er_new[o] = 0;
    }
    __syncthreads();
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        u64 er = 0;
        for (int q = 0; q < L; q++) er |= p.pos_er[((size_t)g * L + q) * W + w];
        const u64 a = p.active[g * W + w];
        const u64 nw = ld_cg(p.any_new + g * W + w);
        u64 stop = a & ~er;                                   // NumErasures == 0
        stop |= a & ~nw;                                      // NumErasures == NumErasuresPrec (first iteration: Prec = n)
        if (p.iter + 1 >= p.max_it) stop = a;                 // while (iter < MaxNumIt)
        s_stop[w] = stop;
        s_act[w] = a;
        const u64 left = a & ~stop;
        p.active[g * W + w] = left;
        p.any_new[g * W + w] = 0;
        if (left) s_alive = 1;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_stop[w] >> b) & 1ull) p.iters[g * p.lanes + l] += p.iter + 1;
        if (TRAJ) {
            int dvn = 0, d1 = 0;
            for (int sl = 0; sl < SCLDPC_CNT_SLOTS; sl++) {
                const size_t o = ((size_t)g * SCLDPC_CNT_SLOTS + sl) * p.lanes + l;
                dvn += ld_cg(p.cnt_dvn + o);
                d1 += ld_cg(p.cnt_deg1 + o);
                p.cnt_dvn[o] = 0;
                p.cnt_deg1[o] = 0;
            }
            if (((s_act[w] >> b) & 1ull) && p.row >= 0 && p.row < p.max_rows) {
                int first = L;
                for (int q = 0; q < L; q++)
                    if ((p.pos_er[((size_t)g * L + q) * W + w] >> b) & 1ull) { first = q; break; }
                int *r = p.rows + (((size_t)g * p.max_rows + p.row) * p.lanes + l) * 3;
                r[0] = d1; r[1] = dvn; r[2] = first;
            }
        }
    }
    // lists of the next iteration
    for (int q = threadIdx.x; q < L; q += blockDim.x) s_chg[q] = (ld_cg(p.vn_stamp + g * L + q) == p.iter);
    __syncthreads();
    for (int c = threadIdx.x; c < ncp; c += blockDim.x) {
        unsigned char any = 0;
        if (c < p.cn_pos_lim)
            for (int i = 0; i < p.dv; i++)
                if (c - i >= 0 && c - i < L && s_chg[c - i]) any = 1;
        s_cn[c] = any;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int nc = 0, nv = 0;
        for (int c = 0; c < ncp; c++)
            if (s_cn[c]) p.cn_list[g * ncp + nc++] = c;
        for (int q = 0; q < L; q++) {
            bool any = false;
            for (int i = 0; i < p.dv; i++) any |= (s_cn[q + i] != 0);
            if (any) p.vn_list[g * L + nv++] = q;
        }
        p.swept[2 * g] += p.n_list[2 * g];
        p.swept[2 * g + 1] += n_vn;
        p.n_list[2 * g] = nc;
        p.n_list[2 * g + 1] = nv;
        p.ticket[g] = 0;
        if (!s_alive) { p.alive[g] = 0; atomicSub(p.alive_total, 1); }
    }
}

// ------------------------------------------------------------------------------------------------------------
// variable-node sweep over the listed positions
// ------------------------------------------------------------------------------------------------------------
template <int DV, bool TRAJ>
__global__ void __launch_bounds__(256, TRAJ ? 3 : 4) bp_vn_wave_kernel(BpParams p)
{
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ int s_cnt[TRAJ ? SCLDPC_MAX_LANES : 1];
    __shared__ u128 s_planes[TRAJ ? LC_PLANES * 256 : 1];
    __shared__ u64 s_new[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (TRAJ)
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
    if (threadIdx.x < SCLDPC_MAX_WORDS) s_new[threadIdx.x] = 0;
    __syncthreads();
    LaneCounter lc;
    if (TRAJ) lc.clear();

    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const bool lane_work = nz(act);
    u128 acc_new = zero128();
    const u128 *__restrict__ c2v = p.c2v + (size_t)g * p.nk * p.dc * ch;
    u128 *__restrict__ v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
    const u128 *__restrict__ chan = p.chan + (size_t)g * p.n * ch;
    u128 *__restrict__ x = p.x + (size_t)g * p.n * ch;
    u128 *__restrict__ y = p.y + (size_t)g * p.n * ch;
    const int32_t *__restrict__ vn_slot = p.vn_slot + (size_t)g * p.n * DV;
    const int *__restrict__ list = p.vn_list + g * p.L;

    const int ipp = p.vns_pos << p.chunk_shift;
    const int items = ld_cg(p.n_list + 2 * g + 1) * ipp;
    const int stride = gridDim.x * blockDim.x;
    // The trip count is block-uniform: the row-write decision below is a shuffle over the ch adjacent threads that hold
    // one VN, and in trajectory mode the counter flush is a block-wide step.
    int trip = 0;
    for (int base = blockIdx.x * blockDim.x; base < items; base += stride, trip++) {
        const int idx = base + threadIdx.x;
        const bool work = lane_work && idx < items;
        u128 changed = zero128(), xn = zero128(), yn = zero128(), xo = zero128(), yo = zero128();
        u128 out[DV];
        int v = 0, pos = 0;
        if (work) {
            const int ent = idx / ipp, off = idx - ent * ipp;
            pos = __ldg(list + ent);
            v = pos * p.vns_pos + (off >> p.chunk_shift);
            int s[DV];
            load_row<DV>(vn_slot + (size_t)v * DV, s);
            u128 in[DV];
#pragma unroll
            for (int i = 0; i < DV; i++) in[i] = ld_stream(c2v + (size_t)s[i] * ch + k);
            // After the first iteration the channel value is implied by y: y = 1 needs chan = 1, and a frame with
            // y = 0 has all-zero outgoing messages for good (incoming messages only go 1 -> 0), so chan is not read.
            if (p.first_iter) { yo = ld_stream(chan + (size_t)v * ch + k); xo = ones128(); }
            else { xo = x[(size_t)v * ch + k]; yo = y[(size_t)v * ch + k]; }
            const u128 xdet = p.first_iter ? yo : xo;                      // Lji starts at the channel value
            u128 acc = yo;
#pragma unroll
            for (int i = 0; i < DV; i++) { out[i] = acc; acc &= in[i]; }
            xn = acc;
            acc = ones128();
#pragma unroll
            for (int i = DV - 1; i >= 0; i--) { out[i] &= acc; acc &= in[i]; }
#pragma unroll
            for (int i = 0; i < DV; i++) yn |= out[i];
            changed = make_u128(((xn.x ^ xdet.x) | (yn.x ^ yo.x)) & act.x, ((xn.y ^ xdet.y) | (yn.y ^ yo.y)) & act.y);
        }
        // a VN's row is rewritten when any of its chunks changed (the ch adjacent threads hold one VN)
        unsigned flag = nz(changed) ? 1u : 0u;
        for (int o = 1; o < ch; o <<= 1) flag |= __shfl_xor_sync(0xffffffffu, flag, o);
        if (work) {
            if (p.first_iter || flag) {
                u128 *dst = v2c + ((size_t)v * DV) * ch + k;
#pragma unroll
                for (int i = 0; i < DV; i++) dst[(size_t)i * ch] = out[i];
            }
            if (p.first_iter || neq(xn, xo)) x[(size_t)v * ch + k] = xn;
            if (p.first_iter || neq(yn, yo)) y[(size_t)v * ch + k] = yn;
            if (nz(changed)) {
                int *st = p.vn_stamp + g * p.L + pos;
                if (ld_cg(st) != p.iter) *st = p.iter;
            }
            const u128 newly = xo & ~xn & act;
            acc_new |= newly;
            if (TRAJ) lc.add(newly);
            const u128 er = xn & act;
            if (nz(er)) {
                u64 *pe = p.pos_er_new + ((size_t)g * p.L + pos) * p.W + 2 * k;
                if (er.x & ~ld_cg(pe)) atomicOr(pe, er.x);
                if (er.y & ~ld_cg(pe + 1)) atomicOr(pe + 1, er.y);
            }
        }
        if (TRAJ && (trip % 31) == 30) lane_counter_flush(lc, s_planes, s_cnt, ch);
    }
    if (TRAJ) lane_counter_flush(lc, s_planes, s_cnt, ch);
    acc_new = warp_or_same_chunk(acc_new, ch);
    if ((threadIdx.x & 31) < ch) {
        if (acc_new.x) atomicOr(&s_new[2 * k], acc_new.x);
        if (acc_new.y) atomicOr(&s_new[2 * k + 1], acc_new.y);
    }
    __syncthreads();
    if (threadIdx.x < p.W) {
        const int w = threadIdx.x;
        if (s_new[w] & ~ld_cg(p.any_new + g * p.W + w)) atomicOr(p.any_new + g * p.W + w, s_new[w]);
    }
    if (TRAJ)
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(p.cnt_dvn + ((size_t)g * SCLDPC_CNT_SLOTS + (blockIdx.x % SCLDPC_CNT_SLOTS)) * p.lanes + i, s_cnt[i]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        bp_wave_retire<TRAJ>(p, g);
    }
}

// ------------------------------------------------------------------------------------------------------------
// frame streams: lane recycling
// ------------------------------------------------------------------------------------------------------------
// Frames that share a word finish at very different iterations (eps = 0.49, M = 10000: mean 794, max 1747), and a
// word costs the same whether one or all of its 64 lanes are still decoding.  In stream mode a graph realisation
// decodes a stream of B frames: when a lane's frame stops, its results are harvested and the lane is re-armed with
// the next channel realisation, so (almost) every lane of every word does useful work in every sweep.
//   VN sweep: for lanes in arm_mask the outgoing messages, x and y are (re)initialised from the new frame's channel
//             bits (drawn in place, channel_draw) instead of being computed; such lanes start iterating next sweep.
//   retire  : per-lane iteration counters; stopped lanes go to done_mask and stay untouched (their x is a fixed point).
//   harvest : every few iterations the finalisation kernels run on fail_mask (done with erasures left) only, results are stored under the
//             frame id, and the freed lanes get the next frame ids in ascending lane order (deterministic).
// Only unlimited-iteration decoding streams (a capped frame would keep changing while it waits for the harvest).
// ARM = false is the lean variant for iterations in which no lane takes a new frame (15 of 16).
template <int DV, bool ARM>
__global__ void __launch_bounds__(256, ARM ? 3 : 4) bp_vn_stream_kernel(BpParams p)
{
    // The CN sweep walks graphs and positions upwards; this sweep walks them downwards, so each sweep starts on the rows
    // the other one touched last -- its first gathers (and the x / y rows) are L2 hits instead of HBM reads.
    const int g = graph_of(p, gridDim.y - 1 - blockIdx.y);
    if (ld_cg(p.alive + g) == 0) return;
    __shared__ u64 s_new[SCLDPC_MAX_WORDS], s_er[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (threadIdx.x < SCLDPC_MAX_WORDS) { s_new[threadIdx.x] = 0; s_er[threadIdx.x] = 0; }
    __syncthreads();
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const u128 arm = ARM ? reinterpret_cast<const u128 *>(p.arm_mask)[g * ch + k] : zero128();
    const bool lane_work = nz(act | arm);
    u128 acc_new = zero128(), acc_er = zero128();   // every position is swept, so "an erased VN is left" is a plain OR
    const u128 *__restrict__ c2v = p.c2v + (size_t)g * p.nk * p.dc * ch;
    u128 *__restrict__ v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
    u128 *__restrict__ x = p.x + (size_t)g * p.n * ch;
    u128 *__restrict__ y = p.y + (size_t)g * p.n * ch;
    const int32_t *__restrict__ vn_slot = p.vn_slot + (size_t)g * p.n * DV;
    const int items = p.n << p.chunk_shift;
    const int stride = gridDim.x * blockDim.x;
    const u64 thr = (ARM && nz(arm)) ? p.thr[g] : 0ull;
    const uint64_t gid = p.first_graph + (uint64_t)g;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < items; base += stride) {
        const int idx = base + (threadIdx.x & 31);
        const bool work = lane_work && idx < items;
        u128 changed = zero128(), xn = zero128(), yn = zero128(), xo = zero128(), yo = zero128();
        u128 out[DV];
        // unsigned: the row offsets widen to 64 bits for free (a sign-extended copy of an int row spills at DV = 5, ARM)
        const unsigned v = p.n - 1 - (idx >> p.chunk_shift);
        if (work) {
            int s[DV];
            load_row<DV>(vn_slot + (size_t)v * DV, s);
            u128 in[DV];
#pragma unroll
            for (int i = 0; i < DV; i++) in[i] = ld_stream(c2v + (size_t)s[i] * ch + k);
            xo = x[(size_t)v * ch + k];
            yo = y[(size_t)v * ch + k];
            u128 acc = yo;
#pragma unroll
            for (int i = 0; i < DV; i++) { out[i] = acc; acc &= in[i]; }
            xn = acc;
            acc = ones128();
#pragma unroll
            for (int i = DV - 1; i >= 0; i--) { out[i] &= acc; acc &= in[i]; }
#pragma unroll
            for (int i = 0; i < DV; i++) yn |= out[i];
            if (ARM && nz(arm)) {
                // new frames: Lji = channel value on every edge (BP_FULL.c:913-917), previous decision "all erased"
                const bool forced = p.known && (v % p.vns_pos) < p.known[v / p.vns_pos];
                u128 cw = zero128();
                // freed lanes get consecutive frame ids in ascending lane order, so one Philox call (4 frames) is
                // usually shared by up to four armed lanes
                uint32_t blk = 0xffffffffu, r4[4] = {0, 0, 0, 0};
                for (int half = 0; half < 2; half++) {
                    u64 m = half ? arm.y : arm.x, w = 0;
                    while (m && !forced) {
                        const int b = __ffsll((long long)m) - 1;
                        m &= m - 1;
                        const uint32_t fr = (uint32_t)p.lane_frame[g * p.lanes + k * 128 + half * 64 + b];
                        if ((fr >> 2) != blk) {
                            blk = fr >> 2;
                            philox4x32_10((uint32_t)v, blk, (uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)p.seed ^ 0x6368616Eu,
                                          (uint32_t)(p.seed >> 32), r4);
                        }
                        if ((u64)r4[fr & 3] < thr) w |= 1ull << b;
                    }
                    if (half) cw.y = w; else cw.x = w;
                }
#pragma unroll
                for (int i = 0; i < DV; i++) out[i] = sel(arm, cw, out[i]);
                xn = xn | arm;
                yn = sel(arm, cw, yn);
            }
            changed = make_u128(((xn.x ^ xo.x) | (yn.x ^ yo.x)) & act.x, ((xn.y ^ xo.y) | (yn.y ^ yo.y)) & act.y);
            if (ARM) changed |= arm;
        }
        unsigned flag = nz(changed) ? 1u : 0u;
        for (int o = 1; o < ch; o <<= 1) flag |= __shfl_xor_sync(0xffffffffu, flag, o);
        if (work) {
            if (flag) {
                u128 *dst = v2c + ((size_t)v * DV) * ch + k;
#pragma unroll
                for (int i = 0; i < DV; i++) dst[(size_t)i * ch] = out[i];
            }
            if (neq(xn, xo)) x[(size_t)v * ch + k] = xn;
            if (neq(yn, yo)) y[(size_t)v * ch + k] = yn;
            acc_new |= xo & ~xn & act;
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
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- end of the iteration for graph g ----
    __shared__ u64 s_stop[SCLDPC_MAX_WORDS], s_act[SCLDPC_MAX_WORDS];
    const int W = p.W;
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        const u64 er = ld_cg(p.any_er + g * W + w);
        p.any_er[g * W + w] = 0;
        const u64 a = p.active[g * W + w];
        const u64 nw = ld_cg(p.any_new + g * W + w);
        const u64 stop = a & (~er | ~nw);                      // NumErasures == 0  ||  == NumErasuresPrec
        s_stop[w] = stop;
        s_act[w] = a;
        u64 left = a & ~stop;
        if (ARM) { left |= p.arm_mask[g * W + w]; p.arm_mask[g * W + w] = 0; }   // armed lanes start iterating with the next sweep
        p.active[g * W + w] = left;
        p.done_mask[g * W + w] |= stop;
        p.fail_mask[g * W + w] |= stop & er;
        p.any_new[g * W + w] = 0;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_act[w] >> b) & 1ull) p.lane_iter[g * p.lanes + l] += 1;
    }
    if (threadIdx.x == 0) p.ticket[g] = 0;
}

// statistics of frame slot o ([G][B]) into the checkpoint slots [k0, k1) of the [K][G][B] outputs
__device__ __forceinline__ void store_ck_slots(const BpParams &p, size_t o, int k0, int k1, int residual, int blocks, int e_exp, int b_exp)
{
    const size_t GB = (size_t)p.G * p.frames_per_graph;
    for (int k = k0; k < k1; k++) {
        p.s_residual[k * GB + o] = residual;
        p.s_blocks_err[k * GB + o] = blocks;
        p.s_erasures_exp[k * GB + o] = e_exp;
        p.s_blocks_err_exp[k * GB + o] = b_exp;
    }
}

// harvest step 3 (one block per graph): results of the lanes in done_mask, then re-arm them with the next frame ids.
// CKPT (node-state streams with checkpoints): a frame paused at checkpoint k = lane_ck gets its statistics recorded into
// slot k, advances lane_ck and goes back into active -- it is not re-armed, so its next iteration continues from the settled
// planes with the stall test it had.  A frame that stopped fills every slot from lane_ck on: the caps it has not reached are
// at least its stop iteration.
template <bool CKPT>
__global__ void bp_stream_harvest_kernel(BpParams p, int exp_all)
{
    const int g = graph_of(p, blockIdx.x), L = p.L, W = p.W, B = p.frames_per_graph;
    if (ld_cg(p.alive + g) == 0) return;
    const bool stats = p.stream_mode != SM_HEAD;                // streams with stopping-set records store iters only
    __shared__ int s_rank[SCLDPC_MAX_WORDS + 1];
    __shared__ u64 s_done[SCLDPC_MAX_WORDS], s_arm[SCLDPC_MAX_WORDS];
    __shared__ u64 s_pause[CKPT ? SCLDPC_MAX_WORDS : 1];
    __shared__ int s_frames;
    __shared__ unsigned long long s_its;
    // (the word loops of this kernel run one word per thread: as thread-0 loops they were chains of dependent global round trips,
    // two thirds of the kernel's 21 us)
    if (threadIdx.x < W) { s_done[threadIdx.x] = p.done_mask[g * W + threadIdx.x]; s_arm[threadIdx.x] = 0; }
    if (CKPT && threadIdx.x < W) s_pause[threadIdx.x] = p.pause_mask[g * W + threadIdx.x];
    if (threadIdx.x == 0) { s_frames = 0; s_its = 0; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int r = 0;
        for (int w = 0; w < W; w++) { s_rank[w] = r; r += __popcll(s_done[w]); }
        s_rank[W] = r;
    }
    __syncthreads();
    const int next0 = p.next_frame[g];
    // frames that stopped with erased VNs left (fail_mask): one warp per frame sums the per-position counts; every other
    // frame's counts are zero by construction
    for (int l = threadIdx.x >> 5; l < p.lanes; l += blockDim.x >> 5) {
        const int w = l >> 6, b = l & 63;
        const u64 counted = CKPT ? (s_done[w] | s_pause[w]) : s_done[w];
        if (!((counted >> b) & 1ull) || !((p.fail_mask[g * W + w] >> b) & 1ull)) continue;
        const int fr = p.lane_frame[g * p.lanes + l];
        int residual = 0, blocks = 0, e_exp = 0, b_exp = 0, first_q = INT_MAX, first_ex = 0;
        for (int q = threadIdx.x & 31; q < L; q += 32) {
            const size_t o = ((size_t)g * L + q) * p.lanes + l;
            const int plain = p.pos_cnt[o], ex = plain - 2 * p.pos_pairs[o];
            if (plain) p.pos_cnt[o] = 0;
            if (plain != ex) p.pos_pairs[o] = 0;
            residual += plain;
            if (plain > 0) blocks++;
            if (ex > 0) {
                e_exp += ex; b_exp++;
                if (first_q == INT_MAX) { first_q = q; first_ex = ex; }     // q ascends within a thread
            }
        }
        if (!exp_all) {                                          // decodeBP adds only the first such position (BP_FULL.c:1126-1131)
            int fq = first_q;
            for (int o = 16; o; o >>= 1) fq = min(fq, __shfl_xor_sync(0xffffffffu, fq, o));
            e_exp = (fq != INT_MAX && first_q == fq) ? first_ex : 0;
            b_exp = (fq != INT_MAX && first_q == fq) ? 1 : 0;
        }
        for (int o = 16; o; o >>= 1) {
            residual += __shfl_xor_sync(0xffffffffu, residual, o);
            blocks += __shfl_xor_sync(0xffffffffu, blocks, o);
            e_exp += __shfl_xor_sync(0xffffffffu, e_exp, o);
            b_exp += __shfl_xor_sync(0xffffffffu, b_exp, o);
        }
        if ((threadIdx.x & 31) == 0 && fr >= 0 && fr < B && stats) {
            const size_t o = (size_t)g * B + fr;
            if (CKPT) {
                const int k0 = p.lane_ck[g * p.lanes + l];
                store_ck_slots(p, o, k0, ((s_pause[w] >> b) & 1ull) ? k0 + 1 : p.n_caps, residual, blocks, e_exp, b_exp);
            } else {
                p.s_residual[o] = residual;
                p.s_blocks_err[o] = blocks;
                p.s_erasures_exp[o] = e_exp;
                p.s_blocks_err_exp[o] = b_exp;
            }
        }
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if (CKPT && ((s_pause[w] >> b) & 1ull)) {              // paused: snapshot without erasures, next checkpoint, resume
            const int fr = p.lane_frame[g * p.lanes + l], k = p.lane_ck[g * p.lanes + l];
            if (fr >= 0 && fr < B && !((p.fail_mask[g * W + w] >> b) & 1ull)) store_ck_slots(p, (size_t)g * B + fr, k, k + 1, 0, 0, 0, 0);
            p.lane_ck[g * p.lanes + l] = k + 1;
            continue;
        }
        if (!((s_done[w] >> b) & 1ull)) continue;
        const int fr = p.lane_frame[g * p.lanes + l];
        if (fr >= 0 && fr < B) {
            const size_t o = (size_t)g * B + fr;
            int its = p.lane_iter[g * p.lanes + l];
            // node-state streams: a frame that finished was seen to stop one iteration late ("nothing resolved")
            if (p.lazy_success && ((p.noprog[g * W + w] >> b) & 1ull) && !((p.fail_mask[g * W + w] >> b) & 1ull)) its -= 1;
            p.s_iters[o] = its;
            atomicAdd(&s_frames, 1);
            atomicAdd(&s_its, (unsigned long long)its);
            if (!((p.fail_mask[g * W + w] >> b) & 1ull) && stats) {
                if (CKPT) store_ck_slots(p, o, p.lane_ck[g * p.lanes + l], p.n_caps, 0, 0, 0, 0);
                else {
                    p.s_residual[o] = 0;
                    p.s_blocks_err[o] = 0;
                    p.s_erasures_exp[o] = 0;
                    p.s_blocks_err_exp[o] = 0;
                }
            }
        }
        if (CKPT) p.lane_ck[g * p.lanes + l] = 0;
        // freed lanes take the next frame ids in ascending lane order
        const int nf = next0 + s_rank[w] + __popcll(s_done[w] & ((1ull << b) - 1ull));
        if (nf < B) {
            p.lane_frame[g * p.lanes + l] = nf;
            p.lane_iter[g * p.lanes + l] = 0;
            atomicOr(reinterpret_cast<unsigned long long *>(&s_arm[w]), 1ull << b);
        } else p.lane_frame[g * p.lanes + l] = -1;
    }
    __syncthreads();
    __shared__ int s_any;
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    if (threadIdx.x < W) {
        const int w = threadIdx.x;
        u64 act = p.active[g * W + w];
        if (CKPT) {                                             // paused frames are live: they continue with the next iteration
            act |= s_pause[w];
            p.pause_mask[g * W + w] = 0;
        }
        p.done_mask[g * W + w] = 0;
        p.fail_mask[g * W + w] = 0;
        p.arm_mask[g * W + w] = s_arm[w];
        if (s_arm[w] | act) s_any = 1;
        if (p.lazy_success) {                                   // ns_arm_kernel writes the new frames before the next iteration
            p.active[g * W + w] = act | s_arm[w];
            p.noprog[g * W + w] = 0;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int any = s_any;
        const int nn = next0 + s_rank[W];
        p.next_frame[g] = nn < B ? nn : B;
        if (!any) { p.alive[g] = 0; atomicSub(p.alive_total, 1); }
        // hint for the host's harvest period: mean iterations per harvested frame of the fastest graph still decoding
        p.h_cum[2 * g] += s_frames;
        p.h_cum[2 * g + 1] += (long long)s_its;
        if (any && p.h_cum[2 * g] > 0) atomicMin(p.alive_total + 1 + p.harvest_parity, (int)(p.h_cum[2 * g + 1] / p.h_cum[2 * g]));
    }
}

__global__ void bp_stream_init_kernel(BpParams p, int n_lanes_used)
{
    const int g = blockIdx.x;
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        p.lane_frame[g * p.lanes + l] = -1;
        p.lane_iter[g * p.lanes + l] = 0;
    }
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        const int lo = w * 64;
        // every usable lane starts "done" with no frame: the first harvest only arms them
        p.done_mask[g * p.W + w] = (n_lanes_used >= lo + 64) ? ~0ull : (n_lanes_used <= lo ? 0ull : ((1ull << (n_lanes_used - lo)) - 1ull));
        p.arm_mask[g * p.W + w] = 0;
        p.fail_mask[g * p.W + w] = 0;
        p.active[g * p.W + w] = 0;
    }
    if (threadIdx.x == 0) p.next_frame[g] = 0;
}

// ------------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------------
template <int DV, int DC>
static void launch_wave_iteration(const BpParams &p, bool traj, cudaStream_t st)
{
    const int block = 256;
    static int res_cn[2] = {0, 0}, res_vn[2] = {0, 0};
    if (!res_cn[0]) {
        res_cn[0] = resident_blocks(bp_cn_wave_kernel<DC, false>, block);
        res_cn[1] = resident_blocks(bp_cn_wave_kernel<DC, true>, block);
        res_vn[0] = resident_blocks(bp_vn_wave_kernel<DV, false>, block);
        res_vn[1] = resident_blocks(bp_vn_wave_kernel<DV, true>, block);
    }
    // every graph gets enough blocks to fill the machine on its own (one wave: the resident block count): blocks
    // of finished graphs return at once, so the graphs still decoding always have the whole GPU
    auto grid = [&](int resident, long long items_per_graph) {
        long long need = (items_per_graph + block - 1) / block;
        long long gx = need < resident ? need : resident;
        return dim3((unsigned)(gx < 1 ? 1 : gx), (unsigned)p.G, 1);
    };
    dim3 gc = grid(res_cn[traj], (long long)p.cn_pos_lim * p.cns_pos << p.chunk_shift);
    dim3 gv = grid(res_vn[traj], (long long)p.n << p.chunk_shift);
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += 2;
    if (p.cn_dis_lim > 0) bp_cn_wave_kernel<DC, false, true><<<gc, block, 0, st>>>(p);     // error-rate runs only (no trajectory)
    else if (traj) bp_cn_wave_kernel<DC, true><<<gc, block, 0, st>>>(p);
    else bp_cn_wave_kernel<DC, false><<<gc, block, 0, st>>>(p);
    if (sample) cudaEventRecord(ev[1], st);
    if (traj) bp_vn_wave_kernel<DV, true><<<gv, block, 0, st>>>(p);
    else bp_vn_wave_kernel<DV, false><<<gv, block, 0, st>>>(p);
    if (sample) {
        cudaEventRecord(ev[2], st);
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

int bp_launch_wave_iteration(int dv, int dc, const BpParams &p, bool traj, cudaStream_t st)
{
#define CALL_WV(A, B) launch_wave_iteration<A, B>(p, traj, st)
    SCLDPC_DISPATCH(dv, dc, CALL_WV);
#undef CALL_WV
    return 0;
}

template <int DV, int DC>
static void launch_stream_iteration(const BpParams &p, bool arm, cudaStream_t st)
{
    const int block = 256;
    static int res_cn = 0, res_vn_arm = 0, res_vn_lean = 0;
    if (!res_cn) {
        res_cn = resident_blocks(bp_cn_wave_kernel<DC, false>, block);
        res_vn_arm = resident_blocks(bp_vn_stream_kernel<DV, true>, block);
        res_vn_lean = resident_blocks(bp_vn_stream_kernel<DV, false>, block);
    }
    const int res_vn = arm ? res_vn_arm : res_vn_lean;
    auto grid = [&](int resident, long long items_per_graph) {
        long long need = (items_per_graph + block - 1) / block;
        long long gx = need < resident ? need : resident;
        return dim3((unsigned)(gx < 1 ? 1 : gx), graphs_in_grid(p), 1);
    };
    dim3 gc = grid(res_cn, (long long)p.cn_pos_lim * p.cns_pos << p.chunk_shift);
    dim3 gv = grid(res_vn, (long long)p.n << p.chunk_shift);
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += 2;
    bp_cn_wave_kernel<DC, false><<<gc, block, 0, st>>>(p);
    if (sample) cudaEventRecord(ev[1], st);
    if (arm) bp_vn_stream_kernel<DV, true><<<gv, block, 0, st>>>(p);
    else bp_vn_stream_kernel<DV, false><<<gv, block, 0, st>>>(p);
    if (sample) {
        cudaEventRecord(ev[2], st);
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

// arm: lanes re-armed by the preceding harvest take their new frames in this iteration's VN sweep
int bp_launch_stream_iteration(int dv, int dc, const BpParams &p, bool arm, cudaStream_t st)
{
#define CALL_ST(A, B) launch_stream_iteration<A, B>(p, arm, st)
    SCLDPC_DISPATCH(dv, dc, CALL_ST);
#undef CALL_ST
    return 0;
}

void bp_launch_stream_init(const BpParams &p, int n_lanes_used, cudaStream_t st)
{
    g_prof.launches += 1;
    bp_stream_init_kernel<<<p.G, 256, 0, st>>>(p, n_lanes_used);
}

void bp_launch_stream_harvest(const BpParams &p, int exp_all, cudaStream_t st)
{
    g_prof.launches += 1;
    // one warp per failed frame: 32 at a time
    if (p.stream_mode == SM_CKPT) bp_stream_harvest_kernel<true><<<graphs_in_grid(p), 1024, 0, st>>>(p, exp_all);
    else bp_stream_harvest_kernel<false><<<graphs_in_grid(p), 1024, 0, st>>>(p, exp_all);
}

void bp_launch_wave_init(const BpParams &p, cudaStream_t st)
{
    g_prof.launches += 1;
    bp_wave_init_kernel<<<p.G, 128, 0, st>>>(p);
}

}  // namespace scldpc
