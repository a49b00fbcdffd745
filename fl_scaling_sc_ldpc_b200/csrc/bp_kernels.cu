// bp_kernels.cu -- bit-sliced flooding BP over the BEC for (dv,dc)-regular SC-LDPC graphs, sm_100a.
//
// One 64-bit lane word carries the same message in 64 independent frames that share a graph realisation; a thread
// owns one 16-byte chunk (128 frames) of one node.  Message rules are the integer rules of the reference:
//   CN:  Lij[c][j] = OR_{l != j} Lji[.]                         (BP_FULL.c:943-968)
//   VN:  Lji[v][i] = chan[v] AND_{l != i} Lij[.]                (BP_FULL.c:985-1005)
//   dec: VNerased[v] = chan[v] AND_l Lij[.]                     (BP_FULL.c:1009-1034)
// Flooding order is kept (a CN sweep reads only Lji and writes only Lij, a VN sweep the reverse; two launches per
// iteration), so every message equals the reference's at every iteration.
//
// Layout in HBM (per graph g; chunks = n_words/2):
//   v2c  [E+1][chunks] u128   VN-major (row v*dv+i), written coalesced by the VN sweep, gathered by the CN sweep
//   c2v  [nk*dc][chunks] u128 CN-major (row c*dc+j), written coalesced by the CN sweep, gathered by the VN sweep
//   chan [n][chunks], x [n][chunks] (a-posteriori erasures), latch [nk][chunks] (CNresolved, trajectory mode)
// A gather fetches n_words*8 contiguous bytes (64 B at n_words = 8), i.e. whole 32 B sectors.
//
// Stopping is decided on the device: every sweep OR-reduces "a VN was resolved in this iteration" and "an erased
// VN is left" per lane (warp shuffles -> shared memory -> one atomicOr per block and word), and the last block of
// the VN sweep (atomic ticket) retires lanes: NumErasures == 0, NumErasures == NumErasuresPrec (messages are
// monotone, so equal counts <=> no VN resolved) or the iteration cap (BP_FULL.c:1044-1065).
#include <cstdlib>

#include "common.cuh"

namespace scldpc {

// ------------------------------------------------------------------------------------------------------------
// initialisation (BP_FULL.c:913-917; BP_SW.c:650-659; BP_TRAJ.c:922-925)
// ------------------------------------------------------------------------------------------------------------
__global__ void bp_init_messages_kernel(BpParams p, int dv, int dc, int trajectory)
{
    const int g = blockIdx.y;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int ch = p.chunks;
    // Lji = channel value on every edge; the dummy row E stays zero
    u128 *v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
    const u128 *chan = p.chan + (size_t)g * p.n * ch;
    for (size_t i = t0; i < (size_t)(p.E + 1) * ch; i += stride) {
        size_t e = i >> p.chunk_shift;
        int k = (int)(i & (ch - 1));
        v2c[i] = (e < (size_t)p.E) ? chan[(e / dv) * ch + k] : zero128();
    }
    // Lij = 1 everywhere (BP_SW.c:655-659).  decodeBP overwrites every swept CN in iteration 0 before any read;
    // CNs it never sweeps (truncated mode) must hold 1 (BP_TRAJ.c:922-925).
    u128 *c2v = p.c2v + (size_t)g * p.nk * dc * ch;
    for (size_t i = t0; i < (size_t)p.nk * dc * ch; i += stride) c2v[i] = ones128();
    if (trajectory) {
        u128 *latch = p.latch + (size_t)g * p.nk * ch;
        for (size_t i = t0; i < (size_t)p.nk * ch; i += stride) latch[i] = zero128();
    }
}

__global__ void bp_init_ctrl_kernel(BpParams p, int n_frames)
{
    const int g = blockIdx.x;
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        int lo = w * 64;
        u64 m = (n_frames >= lo + 64) ? ~0ull : (n_frames <= lo ? 0ull : ((1ull << (n_frames - lo)) - 1ull));
        p.active[g * p.W + w] = m;
        p.any_new[g * p.W + w] = 0;
        p.any_er[g * p.W + w] = 0;
    }
    for (int i = threadIdx.x; i < p.L * p.W; i += blockDim.x) p.pos_er[(size_t)g * p.L * p.W + i] = 0;
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        p.iters[g * p.lanes + l] = 0;
        for (int sl = 0; sl < SCLDPC_CNT_SLOTS; sl++) {
            p.cnt_dvn[((size_t)g * SCLDPC_CNT_SLOTS + sl) * p.lanes + l] = 0;
            p.cnt_deg1[((size_t)g * SCLDPC_CNT_SLOTS + sl) * p.lanes + l] = 0;
        }
        p.work[g * p.lanes + l] = 0;
    }
    for (int i = threadIdx.x; i < p.L * p.lanes; i += blockDim.x) {
        p.pos_cnt[(size_t)g * p.L * p.lanes + i] = 0;
        p.pos_pairs[(size_t)g * p.L * p.lanes + i] = 0;
    }
    if (threadIdx.x == 0) {
        p.ticket[g] = 0;
        p.alive[g] = n_frames > 0 ? 1 : 0;
        if (g == 0) *p.alive_total = n_frames > 0 ? p.G : 0;
    }
}

// start of a window: every valid lane iterates again (BP_SW.c:695-703)
__global__ void bp_window_begin_kernel(BpParams p, int n_frames)
{
    const int g = blockIdx.x;
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        int lo = w * 64;
        u64 m = (n_frames >= lo + 64) ? ~0ull : (n_frames <= lo ? 0ull : ((1ull << (n_frames - lo)) - 1ull));
        p.active[g * p.W + w] = m;
        p.any_new[g * p.W + w] = 0;
        p.any_er[g * p.W + w] = 0;
    }
    if (threadIdx.x == 0) {
        p.ticket[g] = 0;
        p.alive[g] = n_frames > 0 ? 1 : 0;
        if (g == 0) *p.alive_total = n_frames > 0 ? p.G : 0;
    }
}

// ------------------------------------------------------------------------------------------------------------
// check-node sweep
// ------------------------------------------------------------------------------------------------------------
template <int DC, bool TRAJ, bool FREEZE>
__device__ __forceinline__ void bp_cn_sweep_body(const BpParams &p, const int g)
{
    __shared__ int s_cnt[TRAJ ? SCLDPC_MAX_LANES : 1];
    if (TRAJ) {
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
        __syncthreads();
    }
    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    // old messages are only needed for frames that hold a lane but are no longer iterating in this window
    const bool need_old = FREEZE && neq(act, valid_chunk_mask(k, p.n_valid));
    const u128 *__restrict__ v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
    u128 *__restrict__ c2v = p.c2v + (size_t)g * p.nk * DC * ch;
    const int32_t *__restrict__ cn_edge = p.cn_edge + (size_t)g * p.nk * DC;

    if (nz(act)) {
        const long long items = (long long)(p.c1 - p.c0) << p.chunk_shift;
        const long long stride = (long long)gridDim.x * blockDim.x;
        for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += stride) {
            const int c = p.c0 + (int)(idx >> p.chunk_shift);
            int e[DC];
            load_row<DC>(cn_edge + (size_t)c * DC, e);
            u128 in[DC];
#pragma unroll
            for (int j = 0; j < DC; j++) in[j] = ld_stream(v2c + (size_t)e[j] * ch + k);
            // out[j] = OR_{l != j} in[l] by prefix / suffix ORs
            u128 out[DC];
            u128 acc = zero128();
#pragma unroll
            for (int j = 0; j < DC; j++) { out[j] = acc; acc |= in[j]; }
            acc = zero128();
#pragma unroll
            for (int j = DC - 1; j >= 0; j--) { out[j] |= acc; acc |= in[j]; }
            u128 *dst = c2v + ((size_t)c * DC) * ch + k;
            if (FREEZE && need_old) {                           // some frame of this chunk has stopped: keep its messages
#pragma unroll
                for (int j = 0; j < DC; j++) out[j] = sel(act, out[j], dst[(size_t)j * ch]);
            }
#pragma unroll
            for (int j = 0; j < DC; j++) st_stream(dst + (size_t)j * ch, out[j]);
            if (TRAJ) {
                // degree-one counter with latch (BP_FULL.c:935-979): num_out_resolved = #j with out[j] == 0
                u128 one = zero128(), two = zero128();
#pragma unroll
                for (int j = 0; j < DC; j++) {
                    if (e[j] != p.E) { u128 z = ~out[j]; two |= one & z; one |= z; }
                }
                u128 *lp = p.latch + ((size_t)g * p.nk + c) * ch + k;
                const u128 lat = *lp;
                const u128 cnt = one & ~two & ~lat & act;
                const u128 nl = lat | (one & act);
                if (neq(nl, lat)) *lp = nl;
                if (nz(cnt)) sparse_count(s_cnt, k * 128, cnt);
            }
        }
    }
    if (TRAJ) {
        __syncthreads();
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(p.cnt_deg1 + ((size_t)g * SCLDPC_CNT_SLOTS + (blockIdx.x % SCLDPC_CNT_SLOTS)) * p.lanes + i, s_cnt[i]);
    }
}

template <int DC, bool TRAJ, bool FREEZE>
__global__ void __launch_bounds__(256) bp_cn_sweep_kernel(BpParams p)
{
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    bp_cn_sweep_body<DC, TRAJ, FREEZE>(p, g);
}

// (bp_retire_lanes: common.cuh)

// ------------------------------------------------------------------------------------------------------------
// variable-node sweep + decision + stop flags
// ------------------------------------------------------------------------------------------------------------
// the last block to finish (atomic ticket) retires the lanes
template <int DV, bool TRAJ, bool FREEZE>
__device__ __forceinline__ void bp_vn_sweep_body(const BpParams &p, const int g)
{
    __shared__ int s_cnt[TRAJ ? SCLDPC_MAX_LANES : 1];
    __shared__ u64 s_new[SCLDPC_MAX_WORDS], s_er[SCLDPC_MAX_WORDS];
    __shared__ int s_last;
    if (TRAJ)
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
    if (threadIdx.x < SCLDPC_MAX_WORDS) { s_new[threadIdx.x] = 0; s_er[threadIdx.x] = 0; }
    __syncthreads();

    const int ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 act = reinterpret_cast<const u128 *>(p.active)[g * ch + k];
    const bool need_old = FREEZE && neq(act, valid_chunk_mask(k, p.n_valid));
    u128 acc_new = zero128(), acc_er = zero128();

    if (nz(act)) {
        const u128 *__restrict__ c2v_g = p.c2v + (size_t)g * p.nk * p.dc * ch;
        u128 *__restrict__ v2c = p.v2c + (size_t)g * (p.E + 1) * ch;
        const u128 *__restrict__ chan = p.chan + (size_t)g * p.n * ch;
        u128 *__restrict__ x = p.x + (size_t)g * p.n * ch;
        const int32_t *__restrict__ vn_slot = p.vn_slot + (size_t)g * p.n * DV;
        const long long items = (long long)(p.v1 - p.v0) << p.chunk_shift;
        const long long stride = (long long)gridDim.x * blockDim.x;
        for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += stride) {
            const int v = p.v0 + (int)(idx >> p.chunk_shift);
            int s[DV];
            load_row<DV>(vn_slot + (size_t)v * DV, s);
            u128 in[DV];
#pragma unroll
            for (int i = 0; i < DV; i++) in[i] = ld_stream(c2v_g + (size_t)s[i] * ch + k);
            const u128 cv = ld_stream(chan + (size_t)v * ch + k);
            u128 xo = ones128();
            if (!p.first_iter) xo = x[(size_t)v * ch + k];
            // out[i] = chan AND_{l != i} in[l];  xn = chan AND_l in[l]
            u128 out[DV];
            u128 acc = cv;
#pragma unroll
            for (int i = 0; i < DV; i++) { out[i] = acc; acc &= in[i]; }
            u128 xn = acc;
            acc = ones128();
#pragma unroll
            for (int i = DV - 1; i >= 0; i--) { out[i] &= acc; acc &= in[i]; }
            u128 *dst = v2c + ((size_t)v * DV) * ch + k;
            if (FREEZE && need_old) {
#pragma unroll
                for (int i = 0; i < DV; i++) out[i] = sel(act, out[i], dst[(size_t)i * ch]);
                xn = sel(act, xn, xo);
            }
#pragma unroll
            for (int i = 0; i < DV; i++) st_stream(dst + (size_t)i * ch, out[i]);
            if (p.first_iter || neq(xn, xo)) x[(size_t)v * ch + k] = xn;
            const u128 newly = xo & ~xn & act;
            acc_new |= newly;
            acc_er |= xn & act;
            if (TRAJ) {
                if (nz(newly)) sparse_count(s_cnt, k * 128, newly);
                if (nz(xn)) {
                    u64 *pe = p.pos_er + ((size_t)g * p.L + v / p.vns_pos) * p.W + 2 * k;
                    if (xn.x & ~ld_cg(pe)) atomicOr(pe, xn.x);
                    if (xn.y & ~ld_cg(pe + 1)) atomicOr(pe + 1, xn.y);
                }
            }
        }
    }
    // block reduction of the per-lane flags
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
    if (TRAJ)
        for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(p.cnt_dvn + ((size_t)g * SCLDPC_CNT_SLOTS + (blockIdx.x % SCLDPC_CNT_SLOTS)) * p.lanes + i, s_cnt[i]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket + g, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        bp_retire_lanes<TRAJ>(p, g);
    }
}

template <int DV, bool TRAJ, bool FREEZE>
__global__ void __launch_bounds__(256) bp_vn_sweep_kernel(BpParams p)
{
    const int g = blockIdx.y;
    if (ld_cg(p.alive + g) == 0) return;
    bp_vn_sweep_body<DV, TRAJ, FREEZE>(p, g);
}

// ------------------------------------------------------------------------------------------------------------
// window decoder in node-state form (see bp_node_kernels.cu for the formulation).  Two planes per VN and frame:
//   x  = the state the CNs see (what the VN's outgoing messages say; only changes when the VN is swept), and at the end
//        the decision recorded when the VN's position was the window's target;
//   xb = the VN's a-posteriori erasure from everything it has been told so far (channel AND incoming messages), including
//        by CNs of windows that do not sweep the VN -- the out-of-window messages the reference keeps in Lij.
// CN sweep over [c0, c1): a CN with exactly one erased neighbour in x clears it in xb (frames that still iterate in this
// window only: a frame that stopped keeps its state, like FREEZE).  VN sweep over [v0, v1): x := xb, "a decision changed"
// and "an erased VN is left" for the window-wide stall rule (BP_SW.c:791-816), then the same lane retirement as the message
// kernels.  Checked bit for bit against the message kernels, the oracle and the compiled decodeBP_SW (tests/test_bp_parity_gpu.py:
// residual, P1, blocks, expurgated counts, erased VNs; 1920 random cases of a numpy restatement incl. per-window iterations).
// ------------------------------------------------------------------------------------------------------------
// (the node-state window kernels live in bp_window_node_kernels.cu)

// ------------------------------------------------------------------------------------------------------------
// finalisation: per-position erasure counts, size-two stopping sets, per-frame results
// ------------------------------------------------------------------------------------------------------------
// grid (blocks per position, L, G): erased VNs per (position, lane)
__global__ void __launch_bounds__(256) bp_pos_count_kernel(BpParams p)
{
    __shared__ int s_cnt[SCLDPC_MAX_LANES];
    const int g = graph_of(p, blockIdx.z), pos = blockIdx.y, ch = p.chunks;
    for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) s_cnt[i] = 0;
    __syncthreads();
    const u128 *x = p.x + ((size_t)g * p.n + (size_t)pos * p.vns_pos) * ch;
    const int items = p.vns_pos * ch;
    // a thread keeps its chunk (blockDim and the stride are multiples of ch); chunks without a selected lane are skipped.
    // Streams with checkpoints also count the frames paused at a checkpoint.
    u128 mask = p.lane_mask ? reinterpret_cast<const u128 *>(p.lane_mask)[g * ch + (threadIdx.x & (ch - 1))] : ones128();
    if (p.stream_mode == SM_CKPT) mask |= reinterpret_cast<const u128 *>(p.pause_mask)[g * ch + (threadIdx.x & (ch - 1))];
    if (nz(mask))
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += gridDim.x * blockDim.x) {
            const u128 xv = x[idx] & mask;
            if (nz(xv)) sparse_count(s_cnt, (idx & (ch - 1)) * 128, xv);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < p.lanes; i += blockDim.x)
        if (s_cnt[i]) {
            atomicAdd(p.pos_cnt + ((size_t)g * p.L + pos) * p.lanes + i, s_cnt[i]);
            // node-state streams: "stopped with erased VNs left" is found here, not tracked per iteration
            if (p.lazy_success) atomicOr(reinterpret_cast<unsigned long long *>(p.fail_mask + g * p.W + (i >> 6)), 1ull << (i & 63));
        }
}

// Size-two stopping sets (BP_FULL.c:1075-1125): VNs a < b of one position, both erased, b on every CN of a, no
// other erased VN on those CNs.  Bit-sliced prefilter (every CN of a has exactly one other erased neighbour), then
// a per-lane check that it is the same VN b on all CNs.  One count per accepted pair at the position of a.
template <int DV, int DC>
__global__ void __launch_bounds__(256) bp_pairs_kernel(BpParams p)
{
    const int g = blockIdx.y, ch = p.chunks;
    const u128 *x = p.x + (size_t)g * p.n * ch;
    const int32_t *vn_cn = p.vn_cn + (size_t)g * p.n * DV;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const long long items = (long long)p.n << p.chunk_shift;
    const u128 mask = p.lane_mask ? reinterpret_cast<const u128 *>(p.lane_mask)[g * ch + (threadIdx.x & (ch - 1))] : ones128();
    if (!nz(mask)) return;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(idx >> p.chunk_shift), k = (int)(idx & (ch - 1));
        const u128 xa = x[(size_t)a * ch + k] & mask;
        if (!nz(xa)) continue;
        u128 cand = xa;
        for (int i = 0; i < DV && nz(cand); i++) {
            const int c = vn_cn[(size_t)a * DV + i];
            u128 one = zero128(), two = zero128();
            for (int j = 0; j < DC; j++) {
                const int e = cn_edge[(size_t)c * DC + j];
                if (e == p.E) continue;
                const int u = e / DV;
                if (u == a) continue;
                const u128 xu = x[(size_t)u * ch + k];
                two |= one & xu; one |= xu;
            }
            cand &= one & ~two;
        }
        for (int half = 0; half < 2; half++) {
            u64 m = half ? cand.y : cand.x;
            while (m) {
                const int b = __ffsll((long long)m) - 1;
                m &= m - 1;
                const int w = 2 * k + half;
                int partner = -1; bool ok = true;
                for (int i = 0; i < DV && ok; i++) {
                    const int c = vn_cn[(size_t)a * DV + i];
                    for (int j = 0; j < DC; j++) {
                        const int e = cn_edge[(size_t)c * DC + j];
                        if (e == p.E) continue;
                        const int u = e / DV;
                        if (u == a) continue;
                        const u64 xw = reinterpret_cast<const u64 *>(x)[((size_t)u * ch) * 2 + w];
                        if ((xw >> b) & 1ull) { if (partner < 0) partner = u; else if (partner != u) ok = false; }
                    }
                }
                if (ok && partner > a && partner / p.vns_pos == a / p.vns_pos)
                    atomicAdd(p.pos_pairs + ((size_t)g * p.L + a / p.vns_pos) * p.lanes + w * 64 + b, 1);
            }
        }
    }
}

// Stream-mode variant in two passes (the prefilter above gathers dc rows for each of up to dv CNs of every erased VN, i.e.
// several CN sweeps' worth when a stuck wave leaves half the VNs of a frame erased):
//   bp_ex2_kernel   : per CN, "exactly two erased neighbours" among the selected lanes          (one CN sweep)
//   bp_pairs2_kernel: per erased VN a, AND of that plane over its dv CNs, then the same per-lane check as above
template <int DV, int DC>
__global__ void __launch_bounds__(256) bp_ex2_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y), ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);
    const u128 mask = reinterpret_cast<const u128 *>(p.lane_mask)[g * ch + k];
    if (!nz(mask)) return;
    const u128 *xk = p.x + (size_t)g * p.n * ch + k;
    u128 *ex2 = p.ex2 + (size_t)g * p.nk * ch;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const long long items = (long long)p.nk << p.chunk_shift;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx >> p.chunk_shift);
        int e[DC];
        load_row<DC>(cn_edge + (size_t)c * DC, e);
        u128 one = zero128(), two = zero128(), three = zero128();
#pragma unroll
        for (int j = 0; j < DC; j++) {
            const u128 xu = (e[j] != p.E) ? ld_stream(xk + (unsigned)((e[j] / DV) << p.chunk_shift)) : zero128();
            three |= two & xu; two |= one & xu; one |= xu;
        }
        ex2[(size_t)c * ch + k] = two & ~three & mask;
    }
}

template <int DV, int DC>
__global__ void __launch_bounds__(256) bp_pairs2_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y), ch = p.chunks;
    const u128 *x = p.x + (size_t)g * p.n * ch;
    const u128 *ex2 = p.ex2 + (size_t)g * p.nk * ch;
    const int32_t *vn_cn = p.vn_cn + (size_t)g * p.n * DV;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const long long items = (long long)p.n << p.chunk_shift;
    const int k = threadIdx.x & (ch - 1);
    const u128 mask = reinterpret_cast<const u128 *>(p.lane_mask)[g * ch + k];
    if (!nz(mask)) return;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(idx >> p.chunk_shift);
        u128 cand = x[(size_t)a * ch + k] & mask;
        if (!nz(cand)) continue;
        int cs[DV];
        load_row<DV>(vn_cn + (size_t)a * DV, cs);
        // the first CN alone rejects most rows (in a stalled frame about a fifth of the CNs have exactly two erased neighbours), so
        // the other dv-1 gathers wait for it: less than half the rows of the plane the one-shot AND fetched
        cand &= ld_stream(ex2 + (size_t)cs[0] * ch + k);
        if (!nz(cand)) continue;
#pragma unroll
        for (int i = 1; i < DV; i++) cand &= ld_stream(ex2 + (size_t)cs[i] * ch + k);
        for (int half = 0; half < 2; half++) {
            u64 m = half ? cand.y : cand.x;
            while (m) {
                const int b = __ffsll((long long)m) - 1;
                m &= m - 1;
                const int w = 2 * k + half;
                int partner = -1; bool ok = true;
                for (int i = 0; i < DV && ok; i++) {
                    const int c = cs[i];
                    for (int j = 0; j < DC; j++) {
                        const int e = cn_edge[(size_t)c * DC + j];
                        if (e == p.E) continue;
                        const int u = e / DV;
                        if (u == a) continue;
                        const u64 xw = reinterpret_cast<const u64 *>(x)[((size_t)u * ch) * 2 + w];
                        if ((xw >> b) & 1ull) { if (partner < 0) partner = u; else if (partner != u) ok = false; }
                    }
                }
                if (ok && partner > a && partner / p.vns_pos == a / p.vns_pos)
                    atomicAdd(p.pos_pairs + ((size_t)g * p.L + a / p.vns_pos) * p.lanes + w * 64 + b, 1);
            }
        }
    }
}


__global__ void bp_lane_final_kernel(BpParams p, BpFinalOut o)
{
    const int g = blockIdx.y;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= p.lanes) return;
    int residual = 0, blocks = 0, e_exp = 0, b_exp = 0, p1 = 0, first_done = 0;
    for (int q = 0; q < p.L; q++) {
        const int plain = p.pos_cnt[((size_t)g * p.L + q) * p.lanes + l];
        const int ex = plain - 2 * p.pos_pairs[((size_t)g * p.L + q) * p.lanes + l];
        residual += plain;
        if (plain > 0) blocks++;
        if (ex > 0 && (o.exp_all || !first_done)) { first_done = 1; e_exp += ex; b_exp++; }
        if (q >= o.p1_lo && q <= o.p1_hi) p1 += plain;
    }
    const int idx = g * p.lanes + l;
    o.residual[idx] = residual;
    o.blocks_err[idx] = blocks;
    o.erasures_exp[idx] = e_exp;
    o.blocks_err_exp[idx] = b_exp;
    if (o.erasures_p1) o.erasures_p1[idx] = p1;
}

// ------------------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------------------
template <int DV, int DC>
static void launch_iteration(const BpParams &p, bool traj, bool freeze, cudaStream_t st)
{
    const int block = 256;
    dim3 gc = sweep_grid((long long)(p.c1 - p.c0) << p.chunk_shift, p.G, block, SWEEP_BLOCKS_PER_SM);
    dim3 gv = sweep_grid((long long)(p.v1 - p.v0) << p.chunk_shift, p.G, block, SWEEP_BLOCKS_PER_SM);
    const bool sample = g_prof.sample_every > 0 && g_prof.n_samples < g_prof.max_samples && (p.iter % g_prof.sample_every) == 0;
    cudaEvent_t *ev = sample ? g_prof.ev + 3 * g_prof.n_samples : nullptr;
    if (sample) cudaEventRecord(ev[0], st);
    g_prof.launches += (p.c1 > p.c0) ? 2 : 1;
    if (p.c1 > p.c0) {
        if (traj) bp_cn_sweep_kernel<DC, true, false><<<gc, block, 0, st>>>(p);
        else if (freeze) bp_cn_sweep_kernel<DC, false, true><<<gc, block, 0, st>>>(p);
        else bp_cn_sweep_kernel<DC, false, false><<<gc, block, 0, st>>>(p);
    }
    if (sample) cudaEventRecord(ev[1], st);
    if (traj) bp_vn_sweep_kernel<DV, true, false><<<gv, block, 0, st>>>(p);
    else if (freeze) bp_vn_sweep_kernel<DV, false, true><<<gv, block, 0, st>>>(p);
    else bp_vn_sweep_kernel<DV, false, false><<<gv, block, 0, st>>>(p);
    if (sample) {
        cudaEventRecord(ev[2], st);
        g_prof.iter_idx[g_prof.n_samples++] = p.iter;
    }
}

template <int DV, int DC>
static void launch_finalize(const BpParams &p, const BpFinalOut &o, cudaStream_t st)
{
    int bx = (p.vns_pos * p.chunks + 255) / 256;
    if (bx > 8) bx = 8;
    g_prof.launches += 3;
    bp_pos_count_kernel<<<dim3(bx, p.L, p.G), 256, 0, st>>>(p);
    dim3 gp = sweep_grid((long long)p.n << p.chunk_shift, p.G, 256, 8);
    bp_pairs_kernel<DV, DC><<<gp, 256, 0, st>>>(p);
    bp_lane_final_kernel<<<dim3((p.lanes + 127) / 128, p.G), 128, 0, st>>>(p, o);
}

int bp_launch_iteration(int dv, int dc, const BpParams &p, bool traj, bool freeze, cudaStream_t st)
{
#define CALL_IT(A, B) launch_iteration<A, B>(p, traj, freeze, st)
    SCLDPC_DISPATCH(dv, dc, CALL_IT);
#undef CALL_IT
    return 0;
}

template <int DV, int DC>
static void launch_count_pairs(const BpParams &p, cudaStream_t st)
{
    // blocks per position: 8 left two thirds of the SMs idle in the streams' harvests (400 blocks of 39 dependent trips each,
    // profiles/r02ze_harvest_kernels_ncu.csv); the pair search takes 8 blocks per SM for the same reason (32 registers)
    int bx = (p.vns_pos * p.chunks + 255) / 256;
    if (bx > (p.lazy_success ? 32 : 8)) bx = p.lazy_success ? 32 : 8;
    if (p.lazy_success) {
        BpParams q = p;
        q.lane_mask = p.done_mask;                              // every stopped frame is counted; the failed ones land in fail_mask
        bp_pos_count_kernel<<<dim3(bx, p.L, graphs_in_grid(p)), 256, 0, st>>>(q);
    } else bp_pos_count_kernel<<<dim3(bx, p.L, graphs_in_grid(p)), 256, 0, st>>>(p);
    if (p.stream_mode == SM_HEAD) {                             // streams with stopping-set records classify instead (ss_launch_stream)
        g_prof.launches += 1;
        return;
    }
    dim3 gp = sweep_grid((long long)p.n << p.chunk_shift, p.G, 256, (p.ex2 && p.lane_mask) ? 8 : 4);
    if (p.ex2 && p.lane_mask) {
        g_prof.launches += 3;
        gp.y = graphs_in_grid(p);                               // streams: only the graphs still decoding
        dim3 ge = sweep_grid((long long)p.nk << p.chunk_shift, p.G, 256, 4);
        ge.y = graphs_in_grid(p);
        bp_ex2_kernel<DV, DC><<<ge, 256, 0, st>>>(p);
        bp_pairs2_kernel<DV, DC><<<gp, 256, 0, st>>>(p);
    } else {
        g_prof.launches += 2;
        bp_pairs_kernel<DV, DC><<<gp, 256, 0, st>>>(p);
    }
}

// erased VNs per (position, lane) and accepted size-two stopping sets, restricted to p.lane_mask
int bp_launch_count_pairs(int dv, int dc, const BpParams &p, cudaStream_t st)
{
#define CALL_CP(A, B) launch_count_pairs<A, B>(p, st)
    SCLDPC_DISPATCH(dv, dc, CALL_CP);
#undef CALL_CP
    return 0;
}

int bp_launch_finalize(int dv, int dc, const BpParams &p, const BpFinalOut &o, cudaStream_t st)
{
#define CALL_FIN(A, B) launch_finalize<A, B>(p, o, st)
    SCLDPC_DISPATCH(dv, dc, CALL_FIN);
#undef CALL_FIN
    return 0;
}

// erased VNs per (position, lane) of an arbitrary plane into `out` ([G][L][lanes], += ; every lane)
void bp_launch_pos_count_of(const BpParams &p, const u128 *plane, int *out, cudaStream_t st)
{
    BpParams q = p;
    q.x = const_cast<u128 *>(plane);
    q.pos_cnt = out;
    q.lane_mask = nullptr;
    q.lazy_success = 0;
    int bx = (p.vns_pos * p.chunks + 255) / 256;
    if (bx > 8) bx = 8;
    g_prof.launches += 1;
    bp_pos_count_kernel<<<dim3(bx, p.L, p.G), 256, 0, st>>>(q);
}

void bp_launch_init(const BpParams &p, int dv, int dc, int trajectory, int n_frames, cudaStream_t st)
{
    dim3 g((unsigned)(num_sms() * 4 / (p.G > 0 ? p.G : 1) + 1), (unsigned)p.G);
    g_prof.launches += 2;
    bp_init_messages_kernel<<<g, 256, 0, st>>>(p, dv, dc, trajectory);
    bp_init_ctrl_kernel<<<p.G, 256, 0, st>>>(p, n_frames);
}

void bp_launch_init_ctrl_only(const BpParams &p, int n_frames, cudaStream_t st)
{
    g_prof.launches += 1;
    bp_init_ctrl_kernel<<<p.G, 256, 0, st>>>(p, n_frames);
}

void bp_launch_window_begin(const BpParams &p, int n_frames, cudaStream_t st)
{
    g_prof.launches += 1;
    bp_window_begin_kernel<<<p.G, 64, 0, st>>>(p, n_frames);
}

}  // namespace scldpc
