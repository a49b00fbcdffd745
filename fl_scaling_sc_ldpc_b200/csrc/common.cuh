// common.cuh -- shared device helpers and the internal parameter block of the BP kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "scldpc.h"

typedef unsigned long long u64;
typedef ulonglong2 u128;   // one 16-byte chunk = 128 bit-sliced frames

#define SCLDPC_MAX_WORDS 16
#define SCLDPC_MAX_LANES (64 * SCLDPC_MAX_WORDS)
// per-lane trajectory counters are spread over this many slots (blockIdx.x % slots) so that the blocks' final atomicAdds do
// not all hit the same 64*W addresses; the retire step sums the slots
#define SCLDPC_CNT_SLOTS 4
// node-state frame streams (bp_node_kernels.cu): geometry of the per-warp resolution lists
#define NS_WARPS 8            // warps per block of the sweep
#define NS_MAX_BLOCKS 640     // blocks per graph of the sweep (>= 4 resident blocks x 148 SMs)
#define NS_WCAP 1024          // least list entries per warp and iteration (capi.cu sizes the regions by the trips a warp makes);
                              // a region that overflows has its iteration caught up by a full pass

__device__ __forceinline__ u128 make_u128(u64 a, u64 b) { u128 r; r.x = a; r.y = b; return r; }
__device__ __forceinline__ u128 operator|(u128 a, u128 b) { return make_u128(a.x | b.x, a.y | b.y); }
__device__ __forceinline__ u128 operator&(u128 a, u128 b) { return make_u128(a.x & b.x, a.y & b.y); }
__device__ __forceinline__ u128 operator~(u128 a) { return make_u128(~a.x, ~a.y); }
__device__ __forceinline__ u128 &operator|=(u128 &a, u128 b) { a.x |= b.x; a.y |= b.y; return a; }
__device__ __forceinline__ u128 &operator&=(u128 &a, u128 b) { a.x &= b.x; a.y &= b.y; return a; }
__device__ __forceinline__ bool nz(u128 a) { return (a.x | a.y) != 0ull; }
__device__ __forceinline__ bool neq(u128 a, u128 b) { return ((a.x ^ b.x) | (a.y ^ b.y)) != 0ull; }
// lanes of `m` take `a`, the others `b`
__device__ __forceinline__ u128 sel(u128 m, u128 a, u128 b) { return make_u128((a.x & m.x) | (b.x & ~m.x), (a.y & m.y) | (b.y & ~m.y)); }
__device__ __forceinline__ u128 zero128() { return make_u128(0ull, 0ull); }
__device__ __forceinline__ u128 ones128() { return make_u128(~0ull, ~0ull); }

// lanes of chunk k (128 lanes) that hold a frame when n_valid frames are in use
__device__ __forceinline__ u128 valid_chunk_mask(int k, int n_valid)
{
    const int lo = k * 128;
    auto w = [&](int base) -> u64 { return n_valid >= base + 64 ? ~0ull : (n_valid <= base ? 0ull : ((1ull << (n_valid - base)) - 1ull)); };
    return make_u128(w(lo), w(lo + 64));
}

// streaming (read-once) global load through the non-coherent path, no L1 allocation
__device__ __forceinline__ u128 ld_stream(const u128 *p)
{
    u128 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0,%1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(u128 *p, u128 v)
{
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(v.x), "l"(v.y) : "memory");
}
__device__ __forceinline__ u64 ld_cg(const u64 *p) { return __ldcg(p); }
__device__ __forceinline__ u128 ld_cg128(const u128 *p)
{
    u128 r;
    asm volatile("ld.global.cg.v2.u64 {%0,%1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ int ld_cg(const int *p) { return __ldcg(p); }
__device__ __forceinline__ uint2 ld_cg_u2(const uint2 *p)
{
    uint2 r;
    asm volatile("ld.global.cg.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_cg_u2(uint2 *p, uint2 v)
{
    asm volatile("st.global.cg.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
// fire-and-forget AND at L2.  atomicAnd() with an unused result sometimes compiles to ATOMG (with a response), not to RED:
// measured +18 us per sweep of the node-state stream kernel (profiles/README.md, round 2).
__device__ __forceinline__ void red_and(unsigned *p, unsigned v)
{
    asm volatile("red.global.and.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// OR-reduce a u128 over the threads of a warp that share (threadIdx.x % chunks); chunks is a power of two <= 8
__device__ __forceinline__ u128 warp_or_same_chunk(u128 v, int chunks)
{
    for (int off = chunks; off < 32; off <<= 1) {
        v.x |= __shfl_xor_sync(0xffffffffu, v.x, off);
        v.y |= __shfl_xor_sync(0xffffffffu, v.y, off);
    }
    return v;
}

// per-lane sparse counting: add 1 to cnt[base + bit] (shared memory) for every set bit of the chunk.
// Written as a plain `red.shared` in PTX: with atomicAdd(ptr, 1) the compiler emits a warp-aggregated ATOMS.POPC.INC
// behind an address-matching loop, which is several times slower here because the lanes' addresses almost never coincide
// (measured: CN sweep of the trajectory mode 560 us -> 170 us).
__device__ __forceinline__ void smem_inc(int *p)
{
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
}
__device__ __forceinline__ void sparse_count(int *cnt, int base, u128 m)
{
    u64 a = m.x;
    while (a) { int b = __ffsll((long long)a) - 1; smem_inc(&cnt[base + b]); a &= a - 1; }
    a = m.y;
    while (a) { int b = __ffsll((long long)a) - 1; smem_inc(&cnt[base + 64 + b]); a &= a - 1; }
}

// ---- per-lane counting without atomics (trajectory mode) -------------------------------------------------------------
// Each thread adds its 128-lane indicator words into bit-sliced carry-save counters (5 planes: up to 31 words); the
// block then transposes through shared memory: every lane's count is summed by exactly one thread over the threads that
// hold the lane's chunk.  Cost is independent of how many bits are set (iteration 0 is dense) and there is no contention.
#define LC_PLANES 5
struct LaneCounter {
    u128 c[LC_PLANES];
    __device__ __forceinline__ void clear()
    {
#pragma unroll
        for (int q = 0; q < LC_PLANES; q++) c[q] = zero128();
    }
    __device__ __forceinline__ void add(u128 w)
    {
#pragma unroll
        for (int q = 0; q < LC_PLANES; q++) {
            const u128 t = c[q] & w;
            c[q].x ^= w.x; c[q].y ^= w.y;
            w = t;
        }
    }
};
// s_planes: LC_PLANES * blockDim.x u128 of shared memory; s_cnt: per-lane totals of the block (lanes ints).
// Must be called by every thread of the block (256 threads); ch = chunks per row (power of two <= 8).
__device__ __forceinline__ void lane_counter_flush(LaneCounter &lc, u128 *s_planes, int *s_cnt, int ch)
{
#pragma unroll
    for (int q = 0; q < LC_PLANES; q++) s_planes[q * blockDim.x + threadIdx.x] = lc.c[q];
    lc.clear();
    __syncthreads();
    const int lanes = 128 * ch;
    const int lpt = lanes >= (int)blockDim.x ? lanes / blockDim.x : 1;       // lanes per thread
    const int l0 = threadIdx.x * lpt;
    if (l0 < lanes) {
        const int kk = l0 >> 7, bit0 = l0 & 127;                              // chunk and first bit inside the chunk
        int cnt[4] = {0, 0, 0, 0};
        const unsigned *pl = reinterpret_cast<const unsigned *>(s_planes);
        for (int src = kk; src < (int)blockDim.x; src += ch) {
#pragma unroll
            for (int q = 0; q < LC_PLANES; q++) {
                const unsigned w32 = pl[(q * blockDim.x + src) * 4 + (bit0 >> 5)] >> (bit0 & 31);
#pragma unroll
                for (int l = 0; l < 4; l++)
                    if (l < lpt) cnt[l] += ((w32 >> l) & 1u) << q;
            }
        }
#pragma unroll
        for (int l = 0; l < 4; l++)
            if (l < lpt) s_cnt[l0 + l] += cnt[l];
    }
    __syncthreads();
}

// Philox4x32-10 (Salmon et al., SC'11) -- counter-based: every (graph, position, socket) / (graph, frame, VN) has its own
// number regardless of how work is split over threads, batches or GPUs.
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t (&out)[4])
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// channel draw of (graph gid, frame f, VN v): erased iff the returned 32-bit number is below eps * 2^32
__host__ __device__ __forceinline__ uint32_t channel_draw(uint64_t seed, uint64_t gid, uint32_t frame, uint32_t v)
{
    uint32_t r[4];
    philox4x32_10(v, frame >> 2, (uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)seed ^ 0x6368616Eu, (uint32_t)(seed >> 32), r);
    return r[frame & 3];
}

// one adjacency row (dc CN edges / dv VN slots) with the widest aligned loads the degree allows
template <int D>
__device__ __forceinline__ void load_row(const int32_t *row, int (&e)[D])
{
    if constexpr (D % 4 == 0) {
#pragma unroll
        for (int q = 0; q < D / 4; q++) {
            int4 t = __ldg(reinterpret_cast<const int4 *>(row) + q);
            e[4 * q] = t.x; e[4 * q + 1] = t.y; e[4 * q + 2] = t.z; e[4 * q + 3] = t.w;
        }
    } else if constexpr (D % 2 == 0) {
#pragma unroll
        for (int q = 0; q < D / 2; q++) {
            int2 t = __ldg(reinterpret_cast<const int2 *>(row) + q);
            e[2 * q] = t.x; e[2 * q + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int q = 0; q < D; q++) e[q] = __ldg(row + q);
    }
}

// Internal parameter block (by value to every BP kernel).
struct BpParams {
    // dimensions
    int dv, dc, n, nk, E, L, vns_pos, cns_pos, G, W, chunks, chunk_shift, lanes;
    int n_valid;              // frames per graph (lanes >= n_valid never hold a frame)
    // graph + channel
    const int32_t *vn_cn;     // [G][n][dv]
    const int32_t *vn_slot;   // [G][n][dv]
    const int32_t *cn_edge;   // [G][nk][dc]
    const u128 *chan;         // [G][n][chunks]
    // state
    u128 *v2c;                // [G][E+1][chunks]  VN-major messages (Lji); row E is the all-zero dummy
    u128 *c2v;                // [G][nk*dc][chunks] CN-major messages (Lij)
    u128 *latch;              // [G][nk][chunks]    CNresolved (trajectory mode)
    u128 *x;                  // [G][n][chunks]     a-posteriori erasures (VNerased)
    u64 *active;              // [G][W] lanes still iterating
    u64 *any_new;             // [G][W] lanes that resolved a VN in this iteration
    u64 *any_er;              // [G][W] lanes with an erased VN left (in the window)
    u64 *pos_er;              // [G][L][W] lanes with an erased VN in position p (trajectory mode)
    unsigned *ticket;         // [G]
    int *alive;               // [G] any active lane
    int *alive_total;         // [8] graphs with an active lane; [1], [2]: smallest mean iterations per harvested frame among the
                              //   graphs still decoding (by harvest parity); [6], [7]: length of glist2 (by harvest parity)
    long long *h_cum;         // [G][2] frame streams: frames harvested so far and the iterations they took
    int harvest_parity;       // frame streams: which of alive_total[1..2] this harvest reports into
    int *cnt_dvn;             // [G][slots][lanes] newly resolved VNs of this iteration (trajectory mode)
    int *cnt_deg1;            // [G][slots][lanes] degree-one CNs of this iteration (trajectory mode)
    int *pos_cnt;             // [G][L][lanes] erased VNs per position (finalisation)
    int *pos_pairs;           // [G][L][lanes] accepted size-two stopping sets per position
    long long *work;          // [G][lanes] edge updates (window decoder)
    // wave tracking (full BP): sweeps visit only positions whose inputs changed
    u128 *y;                  // [G][n][chunks] "some outgoing Lji is an erasure" plane (with x: the VN's output state)
    u64 *pos_er_new;          // [G][L][W] scratch of pos_er for the positions swept in this iteration
    int *vn_stamp;            // [G][L] last iteration in which a VN of the position changed an outgoing message
    int *cn_list;             // [G][L+dv-1] CN positions to sweep
    int *vn_list;             // [G][L] VN positions to sweep
    int *n_list;              // [G][2] lengths of cn_list / vn_list
    int cn_pos_lim;           // CN positions that are ever swept (L+dv-1 terminated, L truncated)
    long long *swept;         // [G][2] CN / VN positions swept, summed over iterations (instrumentation)
    const u64 *lane_mask;     // [G][W] finalisation kernels only look at these lanes (NULL: all lanes)
    u128 *cn_dis;             // [G][cn_dis_lim][chunks] CNs below cn_dis_lim that started with exactly one erased neighbour
    int cn_dis_lim;           //   never resolve it (simulate_sc_ldpc with an ignored head, PD.py:604-605,656); 0 = off
    // frame streams (lane recycling): a finished frame frees its bit lane for the next channel realisation
    u64 *arm_mask;            // [G][W] lanes that take a new frame in the next VN sweep
    u64 *done_mask;           // [G][W] lanes whose frame has stopped and waits to be harvested
    u128 *xb;                 // [G][n][chunks] node-state decoders: second plane (streams: x and xb alternate as read / write plane, bp_node_kernels.cu)
    u128 *ex2;                // [G][nk][chunks] frame streams: "exactly two erased neighbours" plane of the harvest (NULL: one-pass pairs kernel)
    u64 *first_new;           // [G][W] node-state streams: lanes whose new frame has a VN the channel left known
    u64 *noprog;              // [G][W] node-state streams: lanes that stopped because an iteration resolved nothing (see bp_node_kernels.cu)
    int32_t *cn_row;          // [G][nk][dc] node-state streams: x-plane row offset (v << chunk_shift) of each CN edge; absent edges
                              //   point at the all-zero row behind the last graph's plane
    uint2 *nl_list;           // [G][2][nl_rw][nl_stride] node-state sweeps: (32-bit word of the plane, bits cleared) per
                              //   resolution of the previous iteration, one private region per warp of the sweep's grid
    int *nl_cnt;              // [G][2][nl_rw] entries in each region
    int nl_stride;            // entries per region: about 48 per trip of a warp (1.5 per thread and trip; measured ~0.5), at least NS_WCAP
    int nl_cap;               // entries of a region in use (nl_stride; SCLDPC_LIST_CAP lowers it so that tests reach the overflow path)
    int nl_rw;                // regions per graph and parity: 8 warps x blocks of the largest sweep, at most NS_MAX_BLOCKS*NS_WARPS
    int *nl_ovf;              // [G][2] some region overflowed: the other plane catches up by a full pass instead
    const int *glist;         // node-state streams: graphs that were still decoding at the last harvest the host has seen (ascending;
    int n_glist;              //   NULL: all G).  Grids are sized by this list, so finished graphs cost no blocks at all (4 graphs per batch,
                              //   one still decoding: 1776 of 2368 blocks of every iteration launch did nothing but exit, 6 us of 58)
    int *glist2;              // [2][G] the lists written by the last two harvests (by harvest parity); count in alive_total[6 + parity]
    int *gshift;              // [G] node-state streams: log2 of the 128-lane chunks the graph's live frames occupy (chunk_shift until the
                              //   tail of the stream, then lowered by the lane compaction, bp_node_kernels.cu)
    int *cmp_cnt;             // [G] lanes moved by the compaction planned at this harvest (0: none)
    int *cmp_src;             // [G][lanes] compaction: lane i takes the frame of lane cmp_src[i]
    int *nl_last;             // [G] node-state window decoder: last iteration the graph executed in the current window
    u64 *win_known;           // [G][W] node-state window decoder: lanes in which the channel left some VN known
    int traj_node;            // node-state synchronous full BP with trajectory rows (bpw_iter_kernel<.,.,.,TRAJ>): pos_pairs holds the
                              //   erased VNs per (position, lane) while decoding, cnt_dvn slot 0 NumErasuresPrec, cnt_deg1 the deg-1 counts
    int win_lists;            // node-state window decoder: 1 = resolution lists (one launch per iteration, bp_window_node_kernels.cu),
                              //   0 = copy variant (CN sweep + copy of the VN window)
    int lazy_success;         // 1: "no erased VN is left" is not tracked per iteration; a frame that finishes stops one iteration
                              //   later on "nothing resolved" and the harvest takes that iteration off again
    u64 *fail_mask;           // [G][W] subset of done_mask that stopped with erased VNs left (the only lanes the count kernels read)
    int *lane_frame;          // [G][lanes] frame id decoded in the lane, -1 if idle
    int *lane_iter;           // [G][lanes] iterations executed by the lane's current frame
    int *next_frame;          // [G] next frame id of the graph's stream
    const u64 *thr;           // [G] erasure threshold eps * 2^32 of the graph's channel
    const int32_t *known;     // [L] doping: the first known[pos] VNs of a position are known (NULL: none)
    int frames_per_graph;     // stream length B
    int stream_cap;           // frame streams: iteration cap per frame (0: none)
    uint64_t seed, first_graph;
    int *s_iters, *s_residual, *s_blocks_err, *s_erasures_exp, *s_blocks_err_exp;   // [G][B] per-frame results
    // outputs
    int *iters;               // [G][lanes]
    int *rows;                // [G][max_rows][lanes][3]
    int max_rows;
    // per-launch
    int c0, c1, v0, v1;       // CN / VN ranges swept
    int iter;                 // iteration index inside the current loop
    int max_it;               // cap of the current loop
    int first_iter;           // 1: the previous a-posteriori state is "all erased" (NumErasuresPrec = n)
    int stall_at_first;       // 1: the stall test is meaningful at first_iter (the sweep covers all n VNs)
    int row;                  // trajectory row written by this iteration (-1: none)
    long long win_edges;      // edge updates of one iteration of the current sweep ranges
    // frame streams with checkpoints (scldpc_bp_stream_caps): a frame that reaches caps[k] (k < n_caps-1) pauses until the
    // harvest, which records its statistics into slot k and lets it continue; stream_cap is the last cap (INT_MAX: unlimited)
    int n_caps;               // 0: no checkpoints
    int caps[SCLDPC_MAX_CAPS];
    int *lane_ck;             // [G][lanes] index of the next checkpoint of the lane's frame
    u64 *pause_mask;          // [G][W] lanes paused at a checkpoint, waiting for the harvest (left active, not in done_mask)
};

// graph handled by block coordinate b of a grid that is sized by the list of graphs still decoding
__device__ __forceinline__ int graph_of(const BpParams &p, unsigned b) { return p.glist ? p.glist[b] : (int)b; }
static inline unsigned graphs_in_grid(const BpParams &p) { return (unsigned)(p.glist ? p.n_glist : p.G); }

// ---- per-warp resolution lists of the node-state sweeps (bp_node_kernels.cu, bp_window_node_kernels.cu) ----------------
// replay of one warp's region of the previous launch on plane `w` (32-bit words of graph g)
__device__ __forceinline__ void ns_replay_region(const BpParams &p, int g, int par_prev, unsigned *w, int rid, bool zero_count)
{
    const int RW = p.nl_rw;
    int *cntp = p.nl_cnt + (size_t)(g * 2 + par_prev) * RW + rid;
    const int cnt = ld_cg(cntp);
    const uint2 *reg = p.nl_list + ((size_t)(g * 2 + par_prev) * RW + rid) * p.nl_stride;
    // eight independent loads in flight per thread (a region holds ~200 entries): one L2 round trip instead of seven
    constexpr int U = 8;
    for (int i0 = threadIdx.x & 31; i0 < cnt; i0 += 32 * U) {
        uint2 e[U];
#pragma unroll
        for (int u = 0; u < U; u++) e[u] = (i0 + 32 * u < cnt) ? ld_cg_u2(reg + i0 + 32 * u) : make_uint2(0u, 0u);
#pragma unroll
        for (int u = 0; u < U; u++)
            if (e[u].y) red_and(w + e[u].x, ~e[u].y);
    }
    if (zero_count && (threadIdx.x & 31) == 0) *cntp = 0;
}

// catch-up after an overflow: w &= r on rows [i0, i1) of the plane (r is the plane the overflowing launch wrote, complete by now)
__device__ __forceinline__ void ns_catch_up(const u128 *r, u128 *w, int i0, int i1)
{
    for (int i = i0 + blockIdx.x * blockDim.x + threadIdx.x; i < i1; i += gridDim.x * blockDim.x) {
        const u128 rv = ld_cg128(r + i), wv = ld_cg128(w + i);
        const unsigned rr[4] = {(unsigned)rv.x, (unsigned)(rv.x >> 32), (unsigned)rv.y, (unsigned)(rv.y >> 32)};
        const unsigned ww[4] = {(unsigned)wv.x, (unsigned)(wv.x >> 32), (unsigned)wv.y, (unsigned)(wv.y >> 32)};
#pragma unroll
        for (int q = 0; q < 4; q++)
            if (ww[q] & ~rr[q]) red_and(reinterpret_cast<unsigned *>(w + i) + q, rr[q]);
    }
}

// ------------------------------------------------------------------------------------------------------------
// lane retirement, run by the last block of a VN sweep for its graph
// ------------------------------------------------------------------------------------------------------------
template <bool TRAJ>
__device__ __forceinline__ void bp_retire_lanes(const BpParams &p, int g)
{
    __shared__ u64 s_stop[SCLDPC_MAX_WORDS], s_act[SCLDPC_MAX_WORDS];
    __shared__ int s_alive;
    if (threadIdx.x == 0) s_alive = 0;
    __syncthreads();
    for (int w = threadIdx.x; w < p.W; w += blockDim.x) {
        const u64 a = p.active[g * p.W + w];
        const u64 nw = ld_cg(p.any_new + g * p.W + w);
        const u64 er = ld_cg(p.any_er + g * p.W + w);
        u64 stop = a & ~er;                                            // NumErasures == 0
        if (!p.first_iter || p.stall_at_first) stop |= a & ~nw;        // NumErasures == NumErasuresPrec
        if (p.iter + 1 >= p.max_it) stop = a;                          // while (iter < MaxNumIt)
        s_stop[w] = stop;
        s_act[w] = a;
        const u64 left = a & ~stop;
        p.active[g * p.W + w] = left;
        p.any_new[g * p.W + w] = 0;
        p.any_er[g * p.W + w] = 0;
        if (left) s_alive = 1;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < p.lanes; l += blockDim.x) {
        const int w = l >> 6, b = l & 63;
        if ((s_stop[w] >> b) & 1ull) {
            p.iters[g * p.lanes + l] += p.iter + 1;
            p.work[g * p.lanes + l] += (long long)(p.iter + 1) * p.win_edges;
        }
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
                int first = p.L;                                        // first_erased = n => prints L (BP_TRAJ.c:1017,1051)
                for (int q = 0; q < p.L; q++)
                    if ((ld_cg(p.pos_er + ((size_t)g * p.L + q) * p.W + w) >> b) & 1ull) { first = q; break; }
                int *r = p.rows + (((size_t)g * p.max_rows + p.row) * p.lanes + l) * 3;
                r[0] = d1; r[1] = dvn; r[2] = first;
            }
        }
    }
    __syncthreads();
    if (TRAJ)
        for (int i = threadIdx.x; i < p.L * p.W; i += blockDim.x) p.pos_er[(size_t)g * p.L * p.W + i] = 0;
    if (threadIdx.x == 0) {
        p.ticket[g] = 0;
        if (!s_alive) { p.alive[g] = 0; atomicSub(p.alive_total, 1); }
    }
}

// Per-frame result pointers of the finalisation kernels.
struct BpFinalOut {
    int *residual, *blocks_err, *erasures_exp, *blocks_err_exp, *erasures_p1;
    int exp_all;         // decodeBP_SW adds every position (BP_SW.c:903-907); decodeBP only the first (BP_FULL.c:1126-1131)
    int p1_lo, p1_hi;    // positions whose erasures count towards NumErasuresP1 (BP_SW.c:846-847); empty if lo > hi
};

// Parameter block of the peeling kernel (peel_kernels.cu).
struct PeelParams {
    int n, dv, n_cn_all, total_size, num_steps, W, n_frames, G;
    int n_words1, n_l1, n_l2;      // bitmap words, level-1 entries (1024 CNs each), level-2 entries (32768 CNs each)
    int bits_global;               // 1: the bitmap lives in global memory behind the block's CN state
    const int32_t *vn_cn;          // [G][n][dv]
    const u64 *chan;               // [G][n][W]
    u64 *state;                    // [gridDim.x][n_cn_all]  (degree << 32) + id sum
    u64 *next;                     // frames handed out beyond the first one of every warp
    int32_t *r1;                   // [G][n_frames][num_steps+1] or NULL
    int32_t *recovered;            // [G][n_frames]
    int32_t *n_erased;             // [G][n_frames]
    uint64_t seed, first_frame;
};

// Parameter block of the stopping-set kernels (ss_kernels.cu).
struct SsParams {
    int dv, dc, n, nk, E, L, vns_pos, G, W, chunks, chunk_shift, lanes;
    const int32_t *vn_cn;      // [G][n][dv]
    const int32_t *cn_edge;    // [G][nk][dc]
    const u128 *x;             // [G][n][chunks] erased VNs after decoding
    const unsigned char *counted;   // [L] 1: VNs of the position can be lost (PD.py:661-666)
    u128 *ge3;                 // [G][nk][chunks]
    int *pos_lost, *pos_big;   // [G][L][lanes]
    int32_t *out;              // [G][lanes][4]
};

// Programmatic dependent launch: the two node-state kernels of an iteration follow each other ~10^5 times per decode, so the launch
// gap between them is worth hiding.  Every block first waits for the predecessor grid (nothing it wrote is read before
// that), then lets the successor's blocks be scheduled as soon as all blocks of this grid have started; those blocks sit
// in their own griddepcontrol.wait until this grid has completed and flushed.
__device__ __forceinline__ void pdl_wait_then_release()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// first failed launch of this thread since the last scldpc_take_launch_error(); the C ABI turns it into SCLDPC_ECUDA
namespace scldpc {
inline cudaError_t &launch_error_slot()
{
    static thread_local cudaError_t e = cudaSuccess;
    return e;
}
inline cudaError_t take_launch_error()
{
    cudaError_t e = launch_error_slot();
    launch_error_slot() = cudaSuccess;
    return e;
}
}  // namespace scldpc

template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, bool pdl, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
    if (e != cudaSuccess && scldpc::launch_error_slot() == cudaSuccess) scldpc::launch_error_slot() = e;
}

// ---- compile-time degrees ----------------------------------------------------------------------------------------------
// The (dv, dc) pairs the decoders are instantiated for: X(DV, DC, arg) once per pair.
#define SCLDPC_DEGREES(X, arg) X(4, 8, arg) X(3, 6, arg) X(5, 10, arg) X(3, 9, arg) X(4, 12, arg)
// CALL(DV, DC) for the pair (dv, dc); the enclosing function returns -1 if the pair is not instantiated
#define SCLDPC_DISPATCH_CASE_(DV, DC, CALL) if (dv_ == DV && dc_ == DC) { CALL(DV, DC); } else
#define SCLDPC_DISPATCH(dv, dc, CALL)                                  \
    do {                                                               \
        const int dv_ = (dv), dc_ = (dc);                              \
        SCLDPC_DEGREES(SCLDPC_DISPATCH_CASE_, CALL) return -1;         \
    } while (0)

// ---- launch geometry ---------------------------------------------------------------------------------------------------
inline int num_sms()
{
    static const int n = [] {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return sms > 0 ? sms : 148;
    }();
    return n;
}

// blocks of `kernel` resident on the whole device at `block` threads per block
template <typename K>
static int resident_blocks(K kernel, int block)
{
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, 0) != cudaSuccess || occ < 1) occ = 2;
    return occ * num_sms();
}

// grid.x for a grid-stride sweep over `items` threads-worth of work replicated over G graphs:
// a whole number of waves of the machine (multiples of the SM count), capped by the work available.
static inline dim3 sweep_grid(long long items, int G, int block, int blocks_per_sm)
{
    long long need = (items + block - 1) / block;
    long long per_graph = (long long)num_sms() * blocks_per_sm;   // each graph can fill the machine on its own
    long long gx = need < per_graph ? need : per_graph;
    if (gx < 1) gx = 1;
    return dim3((unsigned)gx, (unsigned)G, 1);
}
// blocks per SM of the per-iteration sweeps on sweep_grid (message sweeps, copy variant of the node-state window decoder)
#define SWEEP_BLOCKS_PER_SM 8


namespace scldpc {
// host-side instrumentation shared by the launchers (capi.cu owns the storage).  One instance per host thread: concurrent callers
// neither share the launch counter nor each other's samples
struct Profiler {
    long long launches;          // kernels launched by this library since the last reset
    int sample_every;            // 0 = off; otherwise time the sweeps of every sample_every-th iteration
    int max_samples, n_samples;
    cudaEvent_t *ev;             // 3 events per sample: before CN sweep, between, after VN sweep
    int *iter_idx;
};
extern thread_local Profiler g_prof;
}  // namespace scldpc
