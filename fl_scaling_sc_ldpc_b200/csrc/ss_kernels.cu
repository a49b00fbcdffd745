// ss_kernels.cu -- stopping-set bookkeeping of simulate_sc_ldpc on the device (sm_100a).
//
// Reference: PD.py:659-691 + extract_stopping_sets (PD.py:1077-1095).  After the peeling fixed point the "lost" VNs of a
// frame (erased VNs of the counted positions) are split into connected components of the residual graph (two lost VNs are
// connected when they share a CN); the bookkeeping only asks, per frame,
//     num_lost, any component with more than two VNs?, VNs in such components, VN positions touched by such components.
// "Component of v has at most two VNs" is a local predicate: the lost neighbours of v are none, or a single u whose only
// lost neighbour is v.  So no union-find is needed:
//   ss_ge3_kernel      (CN sweep, bit-sliced)  plane "this CN has three or more lost neighbours"
//   ss_classify_kernel (VN sweep)              a lost VN on such a CN is in a big component (bit-sliced, the common case: a
//                                              stuck wave leaves thousands of lost VNs); the few others are checked lane
//                                              by lane by walking their CNs (at most 2 x dv x dc bit tests)
//   ss_final_kernel                            per frame: sums over positions
// Round 1 did this on the host (SciPy connected components, one device-to-host sync per failed frame).
#include "common.cuh"

#include <cstring>

namespace scldpc {

template <int DV, int DC>
__global__ void __launch_bounds__(256) ss_ge3_kernel(SsParams p)
{
    const int g = p.glist ? p.glist[blockIdx.y] : (int)blockIdx.y, ch = p.chunks;
    const int k = threadIdx.x & (ch - 1);                       // a thread keeps its chunk
    if (p.lane_mask && !nz(reinterpret_cast<const u128 *>(p.lane_mask)[g * ch + k])) return;
    const u128 *xk = p.x + (size_t)g * p.n * ch + k;
    u128 *ge3 = p.ge3 + (size_t)g * p.nk * ch;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    const long long items = (long long)p.nk << p.chunk_shift;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx >> p.chunk_shift);
        int e[DC];
        load_row<DC>(cn_edge + (size_t)c * DC, e);
        u128 one = zero128(), two = zero128(), three = zero128();
#pragma unroll
        for (int j = 0; j < DC; j++) {
            u128 xu = zero128();
            if (e[j] != p.E) {
                const int u = e[j] / DV;
                if (p.counted[u / p.vns_pos]) xu = xk[(size_t)u << p.chunk_shift];
            }
            three |= two & xu; two |= one & xu; one |= xu;
        }
        ge3[(size_t)c * ch + k] = three;
    }
}

// the single lost neighbour of VN a in lane (w, b): -1 none, -2 two or more distinct ones
template <int DV, int DC>
__device__ __forceinline__ int ss_lost_neighbour(const SsParams &p, const int32_t *vn_cn, const int32_t *cn_edge, const u64 *xw,
                                                 int a, int w, int b)
{
    int first = -1;
    for (int i = 0; i < DV; i++) {
        const int c = vn_cn[(size_t)a * DV + i];
        for (int j = 0; j < DC; j++) {
            const int e = cn_edge[(size_t)c * DC + j];
            if (e == p.E) continue;
            const int u = e / DV;
            if (u == a || !p.counted[u / p.vns_pos]) continue;
            if ((xw[((size_t)u * p.chunks) * 2 + w] >> b) & 1ull) {
                if (first < 0) first = u;
                else if (first != u) return -2;
            }
        }
    }
    return first;
}

// grid (blocks per position, L, G)
template <int DV, int DC>
__global__ void __launch_bounds__(256) ss_classify_kernel(SsParams p)
{
    __shared__ int s_lost[SCLDPC_MAX_LANES], s_big[SCLDPC_MAX_LANES];
    const int g = p.glist ? p.glist[blockIdx.z] : (int)blockIdx.z, pos = blockIdx.y, ch = p.chunks;
    if (!p.counted[pos]) return;
    // a thread keeps its chunk (blockDim and the stride are multiples of ch) and skips it without a selected lane; the mask is
    // re-read where it is used (an L1 hit), so that it holds no registers over the loop
    const u128 *lmask = reinterpret_cast<const u128 *>(p.lane_mask);
    const int items = (!lmask || nz(lmask[g * ch + (threadIdx.x & (ch - 1))])) ? p.vns_pos * ch : 0;
    for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) { s_lost[i] = 0; s_big[i] = 0; }
    __syncthreads();
    const u128 *x = p.x + (size_t)g * p.n * ch;
    const u64 *xw = reinterpret_cast<const u64 *>(x);
    const u128 *ge3 = p.ge3 + (size_t)g * p.nk * ch;
    const int32_t *vn_cn = p.vn_cn + (size_t)g * p.n * DV;
    const int32_t *cn_edge = p.cn_edge + (size_t)g * p.nk * DC;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < items; idx += gridDim.x * blockDim.x) {
        const int a = pos * p.vns_pos + (idx >> p.chunk_shift), k = idx & (ch - 1);
        u128 xa = x[(size_t)a * ch + k];
        if (lmask) xa &= lmask[g * ch + k];
        if (!nz(xa)) continue;
        int cs[DV];
        load_row<DV>(vn_cn + (size_t)a * DV, cs);
        u128 big = zero128();
#pragma unroll
        for (int i = 0; i < DV; i++) big |= ge3[(size_t)cs[i] * ch + k];
        big &= xa;
        const u128 rest = xa & ~big;
        u128 small = zero128();
        for (int half = 0; half < 2; half++) {
            u64 m = half ? rest.y : rest.x, sm = 0;
            while (m) {
                const int b = __ffsll((long long)m) - 1;
                m &= m - 1;
                const int w = 2 * k + half;
                const int u = ss_lost_neighbour<DV, DC>(p, vn_cn, cn_edge, xw, a, w, b);
                bool is_small = (u == -1);
                if (u >= 0) is_small = ss_lost_neighbour<DV, DC>(p, vn_cn, cn_edge, xw, u, w, b) >= 0;   // then it is a
                if (is_small) sm |= 1ull << b;
            }
            if (half) small.y = sm; else small.x = sm;
        }
        sparse_count(s_lost, k * 128, xa);
        const u128 bg = xa & ~small;
        if (nz(bg)) sparse_count(s_big, k * 128, bg);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < p.lanes; i += blockDim.x) {
        if (s_lost[i]) atomicAdd(p.pos_lost + ((size_t)g * p.L + pos) * p.lanes + i, s_lost[i]);
        if (s_big[i]) atomicAdd(p.pos_big + ((size_t)g * p.L + pos) * p.lanes + i, s_big[i]);
    }
}

__global__ void ss_final_kernel(SsParams p)
{
    const int g = blockIdx.y;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= p.lanes) return;
    int lost = 0, big = 0, blocks = 0;
    for (int q = 0; q < p.L; q++) {
        lost += p.pos_lost[((size_t)g * p.L + q) * p.lanes + l];
        const int bq = p.pos_big[((size_t)g * p.L + q) * p.lanes + l];
        big += bq;
        blocks += bq > 0;
    }
    int32_t *o = p.out + ((size_t)g * p.lanes + l) * 4;
    o[0] = lost; o[1] = big > 0; o[2] = big; o[3] = blocks;
}

template <int DV, int DC>
static void ss_launch_t(const SsParams &p, cudaStream_t st)
{
    ss_ge3_kernel<DV, DC><<<sweep_grid((long long)p.nk << p.chunk_shift, p.G, 256, 4), 256, 0, st>>>(p);
    int bx = (p.vns_pos * p.chunks + 255) / 256;
    if (bx > 8) bx = 8;
    ss_classify_kernel<DV, DC><<<dim3(bx, p.L, p.G), 256, 0, st>>>(p);
    ss_final_kernel<<<dim3((p.lanes + 127) / 128, p.G), 128, 0, st>>>(p);
    g_prof.launches += 3;
}

int ss_launch(const SsParams &p, cudaStream_t st)
{
#define CALL_SS(A, B) ss_launch_t<A, B>(p, st)
    SCLDPC_DISPATCH(p.dv, p.dc, CALL_SS);
#undef CALL_SS
    return 0;
}

// ---- frame streams with stopping-set records (scldpc_bp_stream_stopping_sets) ----------------------------------------------
// At a harvest, after bp_pos_count_kernel has found the frames that stopped with erasures left (fail_mask): ss_ge3_kernel and
// ss_classify_kernel run on the settled plane for those lanes of the graphs still decoding, then ss_stream_record_kernel writes
// the record of every stopped frame under its frame id -- before bp_stream_harvest_kernel re-arms the lanes and overwrites
// lane_frame.  The per-position accumulators of the consumed lanes are zero again afterwards; a frame that stopped without
// erasures gets (0, 0, 0, 0).
__global__ void ss_stream_record_kernel(BpParams p)
{
    const int g = graph_of(p, blockIdx.y), W = p.W;
    if (ld_cg(p.alive + g) == 0) return;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= p.lanes) return;
    const int w = l >> 6, b = l & 63;
    if (!((p.done_mask[g * W + w] >> b) & 1ull)) return;
    int lost = 0, big = 0, blocks = 0;
    if ((p.fail_mask[g * W + w] >> b) & 1ull)
        for (int q = 0; q < p.L; q++) {                         // as ss_final_kernel
            const size_t o = ((size_t)g * p.L + q) * p.lanes + l;
            const int lq = p.ss_lost[o], bq = p.ss_big[o];
            if (lq) p.ss_lost[o] = 0;
            if (bq) p.ss_big[o] = 0;
            lost += lq;
            big += bq;
            blocks += bq > 0;
        }
    const int fr = p.lane_frame[g * p.lanes + l];
    if (fr >= 0 && fr < p.frames_per_graph) {
        int32_t *o = p.ss_records + ((size_t)g * p.frames_per_graph + fr) * 4;
        o[0] = lost; o[1] = big > 0; o[2] = big; o[3] = blocks;
    }
}

template <int DV, int DC>
static void ss_launch_stream_t(const BpParams &b, cudaStream_t st)
{
    SsParams p;
    memset(&p, 0, sizeof p);
    p.dv = b.dv; p.dc = b.dc; p.n = b.n; p.nk = b.nk; p.E = b.E; p.L = b.L; p.vns_pos = b.vns_pos; p.G = b.G; p.W = b.W;
    p.chunks = b.chunks; p.chunk_shift = b.chunk_shift; p.lanes = b.lanes;
    p.vn_cn = b.vn_cn; p.cn_edge = b.cn_edge; p.x = b.x; p.counted = b.ss_counted;
    p.ge3 = b.ex2;                                              // the pair search's plane: not used in this mode
    p.pos_lost = b.ss_lost; p.pos_big = b.ss_big;
    p.lane_mask = b.fail_mask;
    p.glist = b.glist; p.n_glist = b.n_glist;
    const unsigned gy = graphs_in_grid(b);
    dim3 ge = sweep_grid((long long)p.nk << p.chunk_shift, p.G, 256, 4);
    ge.y = gy;
    ss_ge3_kernel<DV, DC><<<ge, 256, 0, st>>>(p);
    int bx = (p.vns_pos * p.chunks + 255) / 256;
    if (bx > 8) bx = 8;
    ss_classify_kernel<DV, DC><<<dim3(bx, p.L, gy), 256, 0, st>>>(p);
    ss_stream_record_kernel<<<dim3((p.lanes + 255) / 256, gy), 256, 0, st>>>(b);
    g_prof.launches += 3;
}

int ss_launch_stream(const BpParams &p, cudaStream_t st)
{
#define CALL_SS(A, B) ss_launch_stream_t<A, B>(p, st)
    SCLDPC_DISPATCH(p.dv, p.dc, CALL_SS);
#undef CALL_SS
    return 0;
}

}  // namespace scldpc
