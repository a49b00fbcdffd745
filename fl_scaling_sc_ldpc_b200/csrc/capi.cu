// capi.cu -- the C ABI of libscldpc.so (declared in include/scldpc.h).  Host-side orchestration only: argument
// checks, workspace carving, the iteration / window loops and the host-buffer convenience entry point.
#include <cuda_runtime.h>

#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <vector>

#include "common.cuh"
#include "scldpc.h"

namespace scldpc {
int bp_launch_iteration(int dv, int dc, const BpParams &p, bool traj, bool freeze, cudaStream_t st);
int bp_launch_finalize(int dv, int dc, const BpParams &p, const BpFinalOut &o, cudaStream_t st);
void bp_launch_init(const BpParams &p, int dv, int dc, int trajectory, int n_frames, cudaStream_t st);
void bp_launch_window_begin(const BpParams &p, int n_frames, cudaStream_t st);
void bp_launch_init_ctrl_only(const BpParams &p, int n_frames, cudaStream_t st);
int bp_launch_wave_iteration(int dv, int dc, const BpParams &p, bool traj, cudaStream_t st);
void bp_launch_wave_init(const BpParams &p, cudaStream_t st);
int bp_launch_stream_iteration(int dv, int dc, const BpParams &p, bool arm, cudaStream_t st);
int bp_launch_node_iteration(int dv, int dc, const BpParams &p, bool after_harvest, cudaStream_t st);
int bp_launch_node_settle(int dv, int dc, const BpParams &p, cudaStream_t st);
void bp_launch_node_arm(const BpParams &p, cudaStream_t st);
void bp_launch_node_compact(const BpParams &p, cudaStream_t st);
void bp_launch_node_alive_list(const BpParams &p, int parity, cudaStream_t st);
void bp_launch_node_tables(const BpParams &p, cudaStream_t st);
int bp_launch_window_node_iteration(int dv, int dc, const BpParams &p, cudaStream_t st);
void bp_launch_window_node_init(const BpParams &p, cudaStream_t st, bool resume);
int bp_launch_window_node_end(int dv, int dc, const BpParams &p, cudaStream_t st);
void bp_launch_window_node_traj_init(const BpParams &p, cudaStream_t st);
void bp_launch_pos_count_of(const BpParams &p, const u128 *plane, int *out, cudaStream_t st);
void bp_launch_stream_init(const BpParams &p, int n_lanes_used, cudaStream_t st);
void bp_launch_stream_harvest(const BpParams &p, int exp_all, cudaStream_t st);
int bp_launch_count_pairs(int dv, int dc, const BpParams &p, cudaStream_t st);
int graph_build_tables(const int32_t *vn_cn, int32_t *vn_slot, int32_t *cn_edge, int32_t *scratch, int *err_dev, int G,
                       int n, int nk, int dv, int dc, cudaStream_t st);
int graph_generate(int32_t *vn_cn, u64 *keys, int G, int L, int vns_pos, int cns_pos, int dv, int dc, uint64_t seed,
                   uint64_t first_graph, int ensemble, cudaStream_t st, uint32_t first_position = 0);
size_t graph_generate_scratch_words(int G, int L, int vns_pos, int cns_pos, int dv, int dc, int ensemble);
void channel_generate(u64 *chan, int G, int n, int W, int n_frames, int vns_pos, const int32_t *known_dev, double eps,
                      uint64_t seed, uint64_t first_graph, uint32_t first_frame, cudaStream_t st, uint32_t first_vn = 0);
void channel_pack(const uint8_t *bytes_dev, u64 *chan, int G, int n, int W, int F, cudaStream_t st);
void bits_unpack(const u64 *bits, uint8_t *bytes_dev, int G, int n, int W, int F, cudaStream_t st);
void peel_picks_host(uint64_t seed, uint64_t frame_id, int n, uint32_t *out);
int peel_grid(int total_size, long long total_frames, int n_cn_all);
size_t peel_state_words(int n_cn_all, int total_size);
int peel_launch(PeelParams p, int grid, cudaStream_t st);
int ss_launch(const SsParams &p, cudaStream_t st);
void corr_moments_launch(const int32_t *r1, int n_frames, int row_len, int start, int step, int K, long long *acc, cudaStream_t st);
void traj_moments_launch(const int32_t *rows, const int32_t *iters, int G, int max_rows, int lanes, int n_frames, long long *acc,
                         cudaStream_t st);
void peel_variance_launch(const int32_t *r1, int n_frames, int row_len, const double *theory, int S, double M, double *ssq,
                          long long *counts, cudaStream_t st);
}  // namespace scldpc

using namespace scldpc;

namespace scldpc { thread_local Profiler g_prof = {0, 0, 0, 0, nullptr, nullptr}; }

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(SCLDPC_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                               \
    } while (0)
// after a group of kernel launches: the sticky runtime error and the first failed cudaLaunchKernelEx of this thread
#define CU_LAUNCHES()                                                                                         \
    do {                                                                                                      \
        CU(cudaGetLastError());                                                                               \
        CU(scldpc::take_launch_error());                                                                      \
    } while (0)

static int check_dims(const scldpc_dims_t *d)
{
    if (!d) return fail(SCLDPC_EINVAL, "dims is NULL");
    if (d->dv < 2 || d->dc < 2 || d->L < 1 || d->vns_pos < 1 || d->cns_pos < 1 || d->n_graphs < 1)
        return fail(SCLDPC_EINVAL, "non-positive dimension");
    if ((long long)d->vns_pos * d->dv != (long long)d->cns_pos * d->dc)
        return fail(SCLDPC_EINVAL, "vns_pos*dv (%lld) != cns_pos*dc (%lld)", (long long)d->vns_pos * d->dv,
                    (long long)d->cns_pos * d->dc);
    const int W = d->n_words;
    if (W < 2 || W > SCLDPC_MAX_WORDS || (W & (W - 1))) return fail(SCLDPC_EINVAL, "n_words must be 2, 4, 8 or 16");
    if (d->n_frames < 0 || d->n_frames > 64 * W) return fail(SCLDPC_EINVAL, "n_frames out of range");
    if (d->n_graphs > 65535) return fail(SCLDPC_EINVAL, "at most 65535 graphs per batch");
    if ((long long)d->L * d->vns_pos * d->dv >= INT_MAX / 2) return fail(SCLDPC_EINVAL, "graph too large for int32 edge ids");
    return 0;
}

static bool degrees_supported(int dv, int dc)
{
#define PAIR_(A, B, _) || (dv == A && dc == B)
    return false SCLDPC_DEGREES(PAIR_, _);
#undef PAIR_
}

static int have_device()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0)
        return fail(SCLDPC_ECUDA, "no CUDA device available (libscldpc has no CPU fallback)");
    return 0;
}

extern "C" const char *scldpc_last_error(void) { return g_err; }
extern "C" int scldpc_version(void) { return 200; }
#ifndef SCLDPC_SRC_HASH
#define SCLDPC_SRC_HASH "unknown"
#endif
// "src=<sha256 prefix of all sources> built=<date time> cuda=<toolkit version> arch=sm_100a": lets a caller (and
// __graft_entry__.build / tests/test_capi_load.py) prove that the loaded .so was compiled from the sources next to it
extern "C" const char *scldpc_build_info(void)
{
    static char buf[160];
    snprintf(buf, sizeof buf, "src=%s built=%s %s cuda=%d.%d arch=sm_100a", SCLDPC_SRC_HASH, __DATE__, __TIME__, CUDART_VERSION / 1000,
             (CUDART_VERSION % 1000) / 10);
    return buf;
}
extern "C" int scldpc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---- workspace ---------------------------------------------------------------------------------------------
static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

struct Carve {
    char *base;
    size_t off;
    template <typename T>
    T *take(size_t count)
    {
        T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += align_up(count * sizeof(T));
        return p;
    }
};

// test hook: an integer from the environment, clamped to [lo, hi]
static int env_int(const char *name, int dflt, int lo, int hi)
{
    const char *s = getenv(name);
    int v = s ? atoi(s) : dflt;
    return v < lo ? lo : (v > hi ? hi : v);
}

// regions of the per-warp resolution lists: one per warp of the largest sweep grid (items = nodes x chunks, 256 per block)
static size_t list_regions(size_t max_nodes, size_t ch)
{
    size_t blocks = (max_nodes * ch + 255) / 256;
    if (blocks > NS_MAX_BLOCKS) blocks = NS_MAX_BLOCKS;
    if (blocks < 1) blocks = 1;
    return blocks * NS_WARPS;
}

// entries per region: a warp makes `trips` trips of 32 (node, chunk) items per sweep and logs about 0.5 resolutions per item
// in steady state (more in the first iterations of a frame); 48 per trip, rounded up to a power of two, 1024 .. 16384
static size_t list_stride(size_t max_nodes, size_t ch)
{
    const size_t regions = list_regions(max_nodes, ch);
    const size_t trips = (max_nodes * ch + regions * 32 - 1) / (regions * 32);
    size_t s = NS_WCAP;
    while (s < 48 * trips && s < 16384) s <<= 1;
    return s;
}

// internal: workspace of scldpc_bp_stream_caps (per-lane checkpoint state on top of the node-state stream's)
#define F_CAPS_WS 0x10000u

static size_t carve(const scldpc_dims_t *d, uint32_t flags, void *ws, BpParams *p)
{
    const size_t G = d->n_graphs, W = d->n_words, ch = W / 2, lanes = 64 * W;
    const size_t n = (size_t)d->L * d->vns_pos, nk = (size_t)(d->L + d->dv - 1) * d->cns_pos, E = n * d->dv;
    Carve c{static_cast<char *>(ws), 0};
    BpParams q;
    memset(&q, 0, sizeof q);
    // frame streams in node-state form (the default, see scldpc_bp_stream) keep no messages: 2 bits per edge less per frame.
    // The layout depends on the flags alone (never on the environment): a size query and a call with the same flags agree.
    const bool no_msgs = (flags & SCLDPC_F_STREAM) && !(flags & SCLDPC_F_MESSAGES);
    q.v2c = no_msgs ? nullptr : c.take<u128>(G * (E + 1) * ch);
    q.c2v = no_msgs ? nullptr : c.take<u128>(G * nk * d->dc * ch);
    q.latch = (flags & SCLDPC_F_TRAJECTORY) ? c.take<u128>(G * nk * ch) : nullptr;
    q.active = c.take<u64>(G * W);
    q.any_new = c.take<u64>(G * W);
    q.any_er = c.take<u64>(G * W);
    q.pos_er = c.take<u64>(G * d->L * W);
    q.ticket = c.take<unsigned>(G);
    q.alive = c.take<int>(G);
    q.alive_total = c.take<int>(8);
    q.h_cum = c.take<long long>(G * 2);
    q.cnt_dvn = c.take<int>(G * SCLDPC_CNT_SLOTS * lanes);
    q.cnt_deg1 = c.take<int>(G * SCLDPC_CNT_SLOTS * lanes);
    q.pos_cnt = c.take<int>(G * d->L * lanes);
    q.pos_pairs = c.take<int>(G * d->L * lanes);
    q.work = c.take<long long>(G * lanes);
    q.y = no_msgs ? nullptr : c.take<u128>(G * n * ch);
    q.pos_er_new = c.take<u64>(G * d->L * W);
    q.vn_stamp = c.take<int>(G * d->L);
    q.cn_list = c.take<int>(G * (d->L + d->dv - 1));
    q.vn_list = c.take<int>(G * d->L);
    q.n_list = c.take<int>(G * 2);
    q.swept = c.take<long long>(G * 2);
    q.arm_mask = c.take<u64>(G * W);
    q.done_mask = c.take<u64>(G * W);
    q.fail_mask = c.take<u64>(G * W);
    q.lane_frame = c.take<int>(G * lanes);
    q.lane_iter = c.take<int>(G * lanes);
    q.next_frame = c.take<int>(G);
    q.thr = c.take<u64>(G);
    q.known = c.take<int32_t>(d->L);
    if (flags & SCLDPC_F_STREAM) {
        q.x = c.take<u128>(G * n * ch + ch);                          // stream mode owns its decision plane; one all-zero row
        q.xb = c.take<u128>(G * n * ch + ch);                         //   behind the last graph stands in for absent CN edges
        q.ex2 = c.take<u128>(G * nk * ch);
        q.first_new = c.take<u64>(G * W);
        q.glist2 = c.take<int>(2 * G);
        if (no_msgs) {
            const size_t RW = list_regions(nk, ch);
            q.nl_rw = (int)RW;
            q.nl_stride = (int)list_stride(nk, ch);
            q.nl_cap = env_int("SCLDPC_LIST_CAP", q.nl_stride, 1, q.nl_stride);   // test hook: does not change the layout
            q.noprog = c.take<u64>(G * W);
            q.cn_row = c.take<int32_t>(G * nk * d->dc);
            q.nl_list = c.take<uint2>(G * 2 * RW * (size_t)q.nl_stride);
            q.nl_cnt = c.take<int>(G * 2 * RW);
            q.nl_ovf = c.take<int>(G * 2);
            q.gshift = c.take<int>(G);
            q.cmp_cnt = c.take<int>(G);
            q.cmp_src = c.take<int>(G * lanes);
            if (flags & F_CAPS_WS) {
                q.lane_ck = c.take<int>(G * lanes);
                q.pause_mask = c.take<u64>(G * W);
            }
        }
    }
    q.cn_dis = (flags & SCLDPC_F_STREAM) ? nullptr : c.take<u128>(G * nk * ch);   // sized for the largest possible ignored head
    if (!(flags & (SCLDPC_F_STREAM | SCLDPC_F_MESSAGES))) {
        // node-state window decoder / synchronous full BP (bp_window_node_kernels.cu): per-warp resolution lists
        const size_t RW = list_regions(nk > n / 4 ? nk : n / 4, ch);
        q.nl_rw = (int)RW;
        q.nl_stride = (int)list_stride(nk > n / 4 ? nk : n / 4, ch);
        q.nl_cap = env_int("SCLDPC_LIST_CAP", q.nl_stride, 1, q.nl_stride);
        q.noprog = c.take<u64>(G * W);
        q.win_known = c.take<u64>(G * W);
        q.nl_last = c.take<int>(G);
        q.nl_list = c.take<uint2>(G * 2 * RW * (size_t)q.nl_stride);
        q.nl_cnt = c.take<int>(G * 2 * RW);
        q.nl_ovf = c.take<int>(G * 2);
    }
    if (p) *p = q;
    return c.off;
}

extern "C" size_t scldpc_bp_workspace_bytes(const scldpc_dims_t *d, uint32_t flags)
{
    if (check_dims(d)) return 0;
    return carve(d, flags, nullptr, nullptr);
}

static int setup_params(const scldpc_dims_t *d, const scldpc_batch_t *b, uint32_t flags, const scldpc_bp_out_t *out,
                        void *ws, size_t ws_bytes, BpParams *p)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!degrees_supported(d->dv, d->dc)) return fail(SCLDPC_EINVAL, "(dv,dc)=(%d,%d) not instantiated", d->dv, d->dc);
    if (!b || !b->vn_cn_dev || !b->vn_slot_dev || !b->cn_edge_dev || !b->chan_dev) return fail(SCLDPC_EINVAL, "batch pointer is NULL");
    if (!out || !out->iters_dev || !out->residual_dev || !out->blocks_err_dev || !out->erasures_exp_dev ||
        !out->blocks_err_exp_dev || !out->erased_dev)
        return fail(SCLDPC_EINVAL, "output pointer is NULL");
    if ((flags & SCLDPC_F_TRAJECTORY) && (!out->rows_dev || out->max_rows <= 0))
        return fail(SCLDPC_EINVAL, "trajectory mode needs rows_dev and max_rows > 0");
    if (!ws) return fail(SCLDPC_EINVAL, "workspace is NULL");
    const size_t need = carve(d, flags, nullptr, nullptr);
    if (ws_bytes < need) return fail(SCLDPC_ENOMEM, "workspace too small: %zu < %zu bytes", ws_bytes, need);
    if ((rc = have_device())) return rc;
    carve(d, flags, ws, p);
    p->dv = d->dv; p->dc = d->dc;
    p->n = d->L * d->vns_pos;
    p->nk = (d->L + d->dv - 1) * d->cns_pos;
    p->E = p->n * d->dv;
    p->L = d->L; p->vns_pos = d->vns_pos; p->cns_pos = d->cns_pos;
    p->G = d->n_graphs; p->W = d->n_words; p->chunks = d->n_words / 2; p->lanes = 64 * d->n_words;
    p->n_valid = d->n_frames;
    p->chunk_shift = 0;
    while ((1 << p->chunk_shift) < p->chunks) p->chunk_shift++;
    p->vn_cn = b->vn_cn_dev; p->vn_slot = b->vn_slot_dev; p->cn_edge = b->cn_edge_dev;
    p->chan = reinterpret_cast<const u128 *>(b->chan_dev);
    p->x = reinterpret_cast<u128 *>(out->erased_dev);
    p->iters = out->iters_dev;
    p->rows = out->rows_dev;
    p->max_rows = out->rows_dev ? out->max_rows : 0;
    p->row = -1;
    return 0;
}

// pinned flag the host polls
static thread_local int *g_host_flag = nullptr;
static int host_flag(int **out)
{
    if (!g_host_flag) CU(cudaMallocHost(&g_host_flag, 64));
    *out = g_host_flag;
    return 0;
}

// ---- graph / channel ------------------------------------------------------------------------------------------
extern "C" int scldpc_graph_build_tables(const scldpc_dims_t *d, const scldpc_batch_t *b, int32_t *scratch_dev, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!b || !b->vn_cn_dev || !b->vn_slot_dev || !b->cn_edge_dev || !scratch_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int n = d->L * d->vns_pos, nk = (d->L + d->dv - 1) * d->cns_pos;
    int *err_dev = nullptr, *hf = nullptr;
    if ((rc = host_flag(&hf))) return rc;
    CU(cudaMallocAsync(&err_dev, sizeof(int), st));
    graph_build_tables(b->vn_cn_dev, b->vn_slot_dev, b->cn_edge_dev, scratch_dev, err_dev, d->n_graphs, n, nk, d->dv, d->dc, st);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(hf, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaFreeAsync(err_dev, st));
    CU(cudaStreamSynchronize(st));
    if (*hf == 1) return fail(SCLDPC_EGRAPH, "CN index out of range in vn_cn");
    if (*hf == 2) return fail(SCLDPC_EGRAPH, "a CN has more than dc edges");
    return 0;
}

// The same without a host synchronisation: the validity flag (0 = fine, 1 = CN index out of range, 2 = a CN with more than dc
// edges) is left in *err_dev for the caller to read when it next synchronises anyway.  Graphs drawn by scldpc_graph_generate
// are valid by construction; the flag matters for injected graphs.
extern "C" int scldpc_graph_build_tables_async(const scldpc_dims_t *d, const scldpc_batch_t *b, int32_t *scratch_dev, int32_t *err_dev,
                                               void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!b || !b->vn_cn_dev || !b->vn_slot_dev || !b->cn_edge_dev || !scratch_dev || !err_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    const int n = d->L * d->vns_pos, nk = (d->L + d->dv - 1) * d->cns_pos;
    graph_build_tables(b->vn_cn_dev, b->vn_slot_dev, b->cn_edge_dev, scratch_dev, err_dev, d->n_graphs, n, nk, d->dv, d->dc,
                       static_cast<cudaStream_t>(stream));
    CU(cudaGetLastError());
    return 0;
}

extern "C" int scldpc_graph_generate(const scldpc_dims_t *d, int32_t *vn_cn_dev, uint64_t *scratch_dev, uint64_t seed,
                                     uint64_t first_graph_id, int tail_biting, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!vn_cn_dev || !scratch_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    if (graph_generate(vn_cn_dev, reinterpret_cast<u64 *>(scratch_dev), d->n_graphs, d->L, d->vns_pos, d->cns_pos, d->dv,
                       d->dc, seed, first_graph_id, tail_biting, static_cast<cudaStream_t>(stream)))
        return fail(SCLDPC_EINVAL, "cns_pos*dc too large for the key layout, or M not a multiple of cns_pos (protograph)");
    CU(cudaGetLastError());
    return 0;
}

extern "C" int scldpc_graph_generate_at(const scldpc_dims_t *d, int32_t *vn_cn_dev, uint64_t *scratch_dev, uint64_t seed,
                                        uint64_t first_graph_id, uint32_t first_position, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!vn_cn_dev || !scratch_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    if (graph_generate(vn_cn_dev, reinterpret_cast<u64 *>(scratch_dev), d->n_graphs, d->L, d->vns_pos, d->cns_pos, d->dv,
                       d->dc, seed, first_graph_id, 0, static_cast<cudaStream_t>(stream), first_position))
        return fail(SCLDPC_EINVAL, "cns_pos*dc too large for the key layout");
    CU(cudaGetLastError());
    return 0;
}

extern "C" size_t scldpc_graph_generate_scratch_bytes(const scldpc_dims_t *d, int tail_biting)
{
    if (check_dims(d)) return 0;
    return sizeof(u64) * graph_generate_scratch_words(d->n_graphs, d->L, d->vns_pos, d->cns_pos, d->dv, d->dc, tail_biting);
}

// doping description -> per-position count of leading VNs that are known (hard: all of them; soft: int(alpha*M))
static int build_known(const scldpc_dims_t *d, const int32_t *doped_pos_host, int n_doped, const int32_t *soft_pos_host,
                       const int32_t *soft_count_host, int n_soft, std::vector<int32_t> *known)
{
    known->assign(d->L, 0);
    for (int i = 0; i < n_doped; i++) {
        if (doped_pos_host[i] < 0 || doped_pos_host[i] >= d->L) return fail(SCLDPC_EINVAL, "doped position out of range");
        (*known)[doped_pos_host[i]] = d->vns_pos;
    }
    for (int i = 0; i < n_soft; i++) {
        if (soft_pos_host[i] < 0 || soft_pos_host[i] >= d->L) return fail(SCLDPC_EINVAL, "soft-doped position out of range");
        int c = soft_count_host[i] < 0 ? 0 : (soft_count_host[i] > d->vns_pos ? d->vns_pos : soft_count_host[i]);
        if (c > (*known)[soft_pos_host[i]]) (*known)[soft_pos_host[i]] = c;
    }
    return 0;
}

static int channel_generate_impl(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                                 int n_doped, const int32_t *soft_pos_host, const int32_t *soft_count_host, int n_soft,
                                 uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id, uint32_t first_vn_id, void *stream);

extern "C" int scldpc_channel_generate(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                                       int n_doped, const int32_t *soft_pos_host, const int32_t *soft_count_host, int n_soft,
                                       uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id, void *stream)
{
    return channel_generate_impl(d, chan_dev, eps, doped_pos_host, n_doped, soft_pos_host, soft_count_host, n_soft, seed,
                                 first_graph_id, first_frame_id, 0, stream);
}

extern "C" int scldpc_channel_generate_at(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                                          int n_doped, uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id,
                                          uint32_t first_vn_id, void *stream)
{
    return channel_generate_impl(d, chan_dev, eps, doped_pos_host, n_doped, nullptr, nullptr, 0, seed, first_graph_id,
                                 first_frame_id, first_vn_id, stream);
}

static int channel_generate_impl(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                                 int n_doped, const int32_t *soft_pos_host, const int32_t *soft_count_host, int n_soft,
                                 uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id, uint32_t first_vn_id, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!chan_dev) return fail(SCLDPC_EINVAL, "chan_dev is NULL");
    if (!(eps >= 0.0 && eps <= 1.0)) return fail(SCLDPC_EINVAL, "eps must be in [0,1]");
    if (first_frame_id & 3u) return fail(SCLDPC_EINVAL, "first_frame_id must be a multiple of 4");
    if ((rc = have_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t *known_dev = nullptr;
    if (n_doped > 0 || n_soft > 0) {
        std::vector<int32_t> known;
        if ((rc = build_known(d, doped_pos_host, n_doped, soft_pos_host, soft_count_host, n_soft, &known))) return rc;
        CU(cudaMallocAsync(&known_dev, sizeof(int32_t) * d->L, st));
        CU(cudaMemcpyAsync(known_dev, known.data(), sizeof(int32_t) * d->L, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));   // `known` leaves scope below
    }
    channel_generate(reinterpret_cast<u64 *>(chan_dev), d->n_graphs, d->L * d->vns_pos, d->n_words, d->n_frames, d->vns_pos,
                     known_dev, eps, seed, first_graph_id, first_frame_id, st, first_vn_id);
    CU(cudaGetLastError());
    if (known_dev) CU(cudaFreeAsync(known_dev, st));
    return 0;
}

extern "C" int scldpc_channel_pack_host(const scldpc_dims_t *d, const uint8_t *erased_host, uint64_t *chan_dev, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!erased_host || !chan_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t n = (size_t)d->L * d->vns_pos, bytes = (size_t)d->n_graphs * d->n_frames * n;
    uint8_t *tmp = nullptr;
    if (bytes) {
        CU(cudaMallocAsync(&tmp, bytes, st));
        CU(cudaMemcpyAsync(tmp, erased_host, bytes, cudaMemcpyHostToDevice, st));
    }
    channel_pack(tmp, reinterpret_cast<u64 *>(chan_dev), d->n_graphs, (int)n, d->n_words, d->n_frames, st);
    CU(cudaGetLastError());
    if (tmp) CU(cudaFreeAsync(tmp, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

// ---- decoders -------------------------------------------------------------------------------------------------
#define POLL_EVERY 8   // iterations enqueued between two polls of the device's counter of graphs still decoding

// Runs up to `cap` flooding iterations, in chunks of POLL_EVERY.  The device keeps the number of graphs that still have an active
// frame; after each chunk that counter is copied to pinned host memory and the NEXT chunk is enqueued before the
// host waits for the copy, so the GPU never idles on the host.  Sweeps of a finished graph return at once, so the
// overshoot (at most two chunks) costs launch latency only.
static int run_iterations(BpParams *p, int dv, int dc, int cap, bool traj, bool freeze, bool wave, cudaStream_t st, int *launched,
                          bool window_node = false)
{
    int *hf = nullptr, rc;
    if ((rc = host_flag(&hf))) return rc;
    static thread_local cudaEvent_t ev[2] = {nullptr, nullptr};
    if (!ev[0]) {
        CU(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    }
    int it = 0, nchunk = 0;
    bool pending[2] = {false, false};
    while (it < cap) {
        const int todo = (cap - it) < POLL_EVERY ? (cap - it) : POLL_EVERY;
        for (int q = 0; q < todo; q++, it++) {
            p->iter = it;
            p->max_it = cap;
            p->first_iter = (it == 0);
            p->row = traj ? it : -1;
            if (window_node ? bp_launch_window_node_iteration(dv, dc, *p, st)
                            : (wave ? bp_launch_wave_iteration(dv, dc, *p, traj, st) : bp_launch_iteration(dv, dc, *p, traj, freeze, st)))
                return fail(SCLDPC_EINVAL, "unsupported degrees");
        }
        CU_LAUNCHES();
        if (it >= cap) break;
        const int slot = nchunk & 1;
        CU(cudaMemcpyAsync(hf + slot, p->alive_total, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(ev[slot], st));
        pending[slot] = true;
        nchunk++;
        const int prev = nchunk & 1;            // the chunk before the one just enqueued
        if (pending[prev]) {
            CU(cudaEventSynchronize(ev[prev]));
            pending[prev] = false;
            if (hf[prev] == 0) break;
        }
    }
    if (launched) *launched += it;
    return 0;
}

// unscanned_head_cns: CNs [0, unscanned_head_cns) are "unscanned" (simulate_sc_ldpc with is_bounded = False: slots below
// ignored_head_schedule*cns_per_pos are never scanned, PD.py:604-605,656); 0 = off.
extern "C" int scldpc_bp_full(const scldpc_dims_t *d, const scldpc_batch_t *b, int max_it, uint32_t flags,
                              int unscanned_head_cns, const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                              int *iters_launched_host, void *stream)
{
    if (unscanned_head_cns < 0) return fail(SCLDPC_EINVAL, "unscanned_head_cns must be >= 0");
    const int g_unscanned_cns = unscanned_head_cns;
    BpParams p;
    int rc = setup_params(d, b, flags, out, workspace_dev, workspace_bytes, &p);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool traj = flags & SCLDPC_F_TRAJECTORY, term = flags & SCLDPC_F_TERMINATED;
    const int cap = max_it <= 0 ? INT_MAX : max_it;
    // Node-state form (bp_window_node_kernels.cu) unless SCLDPC_F_MESSAGES asks for explicit messages: one window that
    // covers the whole code -- same erased set and stopping at every iteration as the message kernels; with
    // SCLDPC_F_TRAJECTORY the TRAJ variant, which also keeps the degree-one latch and exact per-position erasure counts.
    // Trajectory rows from the node-state sweep pay up to M of a few 10^4 (48 100 against 27 500 frames/s at M = 10^4, cap 175);
    // at M = 10^5 the per-(position, frame) counters see ten times the decrements on the same addresses and the message
    // kernels win (3980 against 3000 frames/s), so very large codes keep them unless SCLDPC_F_NODE_TRAJ insists.
    const bool node = d->n_frames > 0 && !(flags & SCLDPC_F_MESSAGES) &&
                      (!traj || d->vns_pos <= 32768 || (flags & SCLDPC_F_NODE_TRAJ));
    if (node) {
        p.xb = p.y;
        p.win_lists = 1;                         // the sweep covers the whole chain: few rows change per iteration
        p.traj_node = traj ? 1 : 0;
        bp_launch_init_ctrl_only(p, d->n_frames, st);
        bp_launch_window_node_init(p, st, false);
        if (traj) {
            CU(cudaMemsetAsync(p.latch, 0, sizeof(u128) * (size_t)p.G * p.nk * p.chunks, st));
            bp_launch_window_node_traj_init(p, st);
            bp_launch_pos_count_of(p, p.chan, p.pos_pairs, st);          // erased VNs per (position, frame) to start with
        }
    } else bp_launch_init(p, d->dv, d->dc, traj, d->n_frames, st);
    CU(cudaGetLastError());
    p.c0 = 0;
    p.c1 = term ? p.nk : d->L * d->cns_pos;     // cn_lim (BP_TRAJ.c:944-948)
    p.v0 = 0;
    p.v1 = p.n;
    p.stall_at_first = 1;
    p.win_edges = 2ll * p.E;
    int launched = 0;
    // wave tracking (bp_wave_kernels.cu) unless disabled or the chain is longer than its shared-memory bitmaps
    const bool wave = !node && d->L + d->dv - 1 <= 1024 && (!(flags & SCLDPC_F_NO_WAVE) || g_unscanned_cns > 0);
    p.cn_dis_lim = g_unscanned_cns;
    if (g_unscanned_cns > 0 && ((!wave && !node) || traj || g_unscanned_cns > p.nk))
        return fail(SCLDPC_EINVAL, "unscanned head: not available with trajectories or for this chain length");
    p.cn_pos_lim = term ? d->L + d->dv - 1 : d->L;
    if (wave) bp_launch_wave_init(p, st);
    if (d->n_frames > 0 && (rc = run_iterations(&p, d->dv, d->dc, cap, traj, false, wave, st, &launched, node))) return rc;
    if (node && bp_launch_window_node_end(d->dv, d->dc, p, st)) return fail(SCLDPC_EINVAL, "unsupported degrees");
    if (node && traj) CU(cudaMemsetAsync(p.pos_pairs, 0, sizeof(int) * (size_t)p.G * p.L * p.lanes, st));   // back to its role in the finalisation
    BpFinalOut fo{out->residual_dev, out->blocks_err_dev, out->erasures_exp_dev, out->blocks_err_exp_dev, out->erasures_p1_dev,
                  (flags & SCLDPC_F_EXP_ALL) ? 1 : 0, 1, 0};
    if (d->n_frames == 0) CU(cudaMemsetAsync(out->erased_dev, 0, sizeof(u64) * (size_t)p.G * p.n * p.W, st));
    bp_launch_finalize(d->dv, d->dc, p, fo, st);
    CU(cudaGetLastError());
    if (iters_launched_host) *iters_launched_host = launched;
    return 0;
}

extern "C" size_t scldpc_bp_stream_workspace_bytes(const scldpc_dims_t *d, uint32_t flags)
{
    if (check_dims(d)) return 0;
    return carve(d, SCLDPC_F_STREAM | (flags & SCLDPC_F_MESSAGES), nullptr, nullptr);
}

extern "C" size_t scldpc_bp_stream_caps_workspace_bytes(const scldpc_dims_t *d)
{
    if (check_dims(d)) return 0;
    return carve(d, SCLDPC_F_STREAM | F_CAPS_WS, nullptr, nullptr);
}

// Frame stream of scldpc_bp_stream (n_caps == 0: `out` holds the [G][B] results) or scldpc_bp_stream_caps (n_caps >= 1:
// `out` holds iters [G][B] and the [K][G][B] statistics; the caps are validated by the caller).
static int bp_stream_impl(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg, const int32_t *caps,
                          int n_caps, const scldpc_stream_out_t *out, void *workspace_dev, size_t workspace_bytes,
                          long long *iters_launched_host, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!degrees_supported(d->dv, d->dc)) return fail(SCLDPC_EINVAL, "(dv,dc)=(%d,%d) not instantiated", d->dv, d->dc);
    if (!b || !b->vn_cn_dev || !b->vn_slot_dev || !b->cn_edge_dev) return fail(SCLDPC_EINVAL, "batch pointer is NULL");
    if (!cfg || !cfg->eps_host || cfg->frames_per_graph < 1) return fail(SCLDPC_EINVAL, "bad stream configuration");
    if (!out || !out->iters_dev || !out->residual_dev || !out->blocks_err_dev || !out->erasures_exp_dev || !out->blocks_err_exp_dev)
        return fail(SCLDPC_EINVAL, "output pointer is NULL");
    if (d->n_frames < 1) return fail(SCLDPC_EINVAL, "n_frames (lanes used per graph) must be >= 1");
    if ((cfg->flags & SCLDPC_F_MESSAGES) && d->L + d->dv - 1 > 1024) return fail(SCLDPC_EINVAL, "chain too long for the message-passing stream");
    if (!workspace_dev) return fail(SCLDPC_EINVAL, "workspace is NULL");
    // SCLDPC_F_MESSAGES selects the message-passing sweeps (the implementation of record); the default is the node-state
    // formulation of bp_node_kernels.cu, which yields the same erased set at every iteration with ~6x less HBM traffic
    const bool node = !(cfg->flags & SCLDPC_F_MESSAGES);
    const uint32_t wflags = SCLDPC_F_STREAM | (cfg->flags & SCLDPC_F_MESSAGES) | (n_caps > 0 ? F_CAPS_WS : 0u);
    const size_t need = carve(d, wflags, nullptr, nullptr);
    if (workspace_bytes < need) return fail(SCLDPC_ENOMEM, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
    if ((rc = have_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    BpParams p;
    carve(d, wflags, workspace_dev, &p);
    p.dv = d->dv; p.dc = d->dc;
    p.n = d->L * d->vns_pos; p.nk = (d->L + d->dv - 1) * d->cns_pos; p.E = p.n * d->dv;
    p.L = d->L; p.vns_pos = d->vns_pos; p.cns_pos = d->cns_pos;
    p.G = d->n_graphs; p.W = d->n_words; p.chunks = d->n_words / 2; p.lanes = 64 * d->n_words;
    p.n_valid = d->n_frames;
    p.chunk_shift = 0;
    while ((1 << p.chunk_shift) < p.chunks) p.chunk_shift++;
    if (node && ((size_t)p.G * p.n + 1) * p.chunks * 4 >= (size_t)1 << 32)
        return fail(SCLDPC_EINVAL, "batch too large for 32-bit plane offsets: reduce n_graphs");
    p.vn_cn = b->vn_cn_dev; p.vn_slot = b->vn_slot_dev; p.cn_edge = b->cn_edge_dev; p.chan = nullptr;
    p.iters = p.lane_iter;                       // scratch for the shared control initialisation
    p.rows = nullptr; p.max_rows = 0; p.row = -1;
    const bool term = cfg->flags & SCLDPC_F_TERMINATED;
    p.cn_pos_lim = term ? d->L + d->dv - 1 : d->L;
    p.c0 = 0; p.c1 = p.cn_pos_lim * d->cns_pos; p.v0 = 0; p.v1 = p.n;
    p.max_it = INT_MAX; p.first_iter = 0; p.stall_at_first = 1;
    p.frames_per_graph = cfg->frames_per_graph; p.seed = cfg->seed; p.first_graph = cfg->first_graph_id;
    p.stream_cap = cfg->max_it > 0 ? cfg->max_it : 0;
    p.n_caps = n_caps;
    for (int k = 0; k < n_caps; k++) p.caps[k] = caps[k];
    if (n_caps > 0) p.stream_cap = caps[n_caps - 1] > 0 ? caps[n_caps - 1] : INT_MAX;
    p.s_iters = out->iters_dev; p.s_residual = out->residual_dev; p.s_blocks_err = out->blocks_err_dev;
    p.s_erasures_exp = out->erasures_exp_dev; p.s_blocks_err_exp = out->blocks_err_exp_dev;
    p.lane_mask = p.fail_mask;                   // frames that stopped without erasures have all-zero counts already
    p.lazy_success = node ? 1 : 0;
    // per-graph channel thresholds and the doping profile
    std::vector<u64> thr(d->n_graphs);
    for (int g = 0; g < d->n_graphs; g++) {
        const double e = cfg->eps_host[g];
        if (!(e >= 0.0 && e <= 1.0)) return fail(SCLDPC_EINVAL, "eps must be in [0,1]");
        thr[g] = e <= 0.0 ? 0 : (e >= 1.0 ? (1ull << 32) : (u64)(e * 4294967296.0));
    }
    std::vector<int32_t> known;
    const bool doped = cfg->n_doped > 0 || cfg->n_soft > 0;
    if (doped && (rc = build_known(d, cfg->doped_pos_host, cfg->n_doped, cfg->soft_pos_host, cfg->soft_count_host, cfg->n_soft, &known))) return rc;
    CU(cudaMemcpyAsync(const_cast<u64 *>(p.thr), thr.data(), sizeof(u64) * thr.size(), cudaMemcpyHostToDevice, st));
    if (doped) CU(cudaMemcpyAsync(const_cast<int32_t *>(p.known), known.data(), sizeof(int32_t) * d->L, cudaMemcpyHostToDevice, st));
    else p.known = nullptr;
    CU(cudaStreamSynchronize(st));               // host vectors leave scope at return; keep it simple
    if (!node && p.stream_cap > 0) return fail(SCLDPC_EINVAL, "capped frame streams need the node-state sweeps (no SCLDPC_F_MESSAGES)");
    // state: no lane holds a frame yet.  Message sweeps: Lij = 1 (tail CNs of a truncated code are never swept), the rest 0
    const size_t ch = p.chunks, plane = ((size_t)p.G * p.n + 1) * ch;
    CU(cudaMemsetAsync(p.x, 0, sizeof(u128) * plane, st));
    CU(cudaMemsetAsync(p.first_new, 0, sizeof(u64) * (size_t)p.G * p.W, st));
    if (node) {
        const size_t RW = (size_t)p.nl_rw;
        CU(cudaMemsetAsync(p.xb, 0, sizeof(u128) * plane, st));
        CU(cudaMemsetAsync(p.noprog, 0, sizeof(u64) * (size_t)p.G * p.W, st));
        CU(cudaMemsetAsync(p.nl_cnt, 0, sizeof(int) * (size_t)p.G * 2 * RW, st));
        CU(cudaMemsetAsync(p.nl_ovf, 0, sizeof(int) * (size_t)p.G * 2, st));
        CU(cudaMemsetAsync(p.swept, 0, sizeof(long long) * (size_t)p.G * 2, st));        // instrumented builds only
        CU(cudaMemsetAsync(p.pos_er, 0, sizeof(u64) * (size_t)p.G * d->L * p.W, st));
        if (n_caps > 0) {
            CU(cudaMemsetAsync(p.lane_ck, 0, sizeof(int) * (size_t)p.G * p.lanes, st));
            CU(cudaMemsetAsync(p.pause_mask, 0, sizeof(u64) * (size_t)p.G * p.W, st));
        }
        bp_launch_node_tables(p, st);
    } else {
        CU(cudaMemsetAsync(p.c2v, 0xFF, sizeof(u128) * (size_t)p.G * p.nk * d->dc * ch, st));
        CU(cudaMemsetAsync(p.v2c, 0, sizeof(u128) * (size_t)p.G * (p.E + 1) * ch, st));
        CU(cudaMemsetAsync(p.y, 0, sizeof(u128) * (size_t)p.G * p.n * ch, st));
    }
    {
        BpParams q = p;                          // control words, counters, position lists ("every position")
        bp_launch_init_ctrl_only(q, d->n_frames, st);
    }
    if (!node) bp_launch_wave_init(p, st);
    bp_launch_stream_init(p, d->n_frames, st);
    bp_launch_stream_harvest(p, 0, st);          // arms the first frames
    if (node) bp_launch_node_arm(p, st);
    CU_LAUNCHES();
    int *hf = nullptr;
    if ((rc = host_flag(&hf))) return rc;
    static thread_local cudaEvent_t ev[2] = {nullptr, nullptr};
    if (!ev[0]) {
        CU(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    }
    // Harvest period: a harvest costs about as much as two to three iterations (count / pair kernels, channel draws of the
    // re-armed lanes) and a finished frame idles H/2 iterations on average, so the best period is about sqrt(6 x iterations
    // per frame); measured flat between 3.5 and 10 at M = 10000.  harvest_every <= 0: adapt it to the frames harvested so far; > 0: fixed.
    const bool adaptive = cfg->harvest_every <= 0;
    // The period follows the FASTEST graph still decoding: a harvest costs every live graph the same, an idle lane costs a
    // fast graph a larger share of its frame.  Measured flat (profiles/r02h_harvest_period_ab.txt: 5.62 .. 5.82e13
    // edge-updates/s for constants 25 .. 60, following the fastest or the slowest graph).
    constexpr int HARVEST_C10 = 60;                // H = sqrt(HARVEST_C10 / 10 x mean iterations per frame), clamped to [8, 64]
    int H = adaptive ? 16 : cfg->harvest_every;
    CU(cudaMemsetAsync(p.alive_total + 1, 0x7f, 2 * sizeof(int), st));
    CU(cudaMemsetAsync(p.h_cum, 0, sizeof(long long) * 2 * (size_t)p.G, st));
    long long it = 0;
    int nchunk = 0;
    bool pending[2] = {false, false};
    for (;;) {
        for (int q = 0; q < H; q++, it++) {
            p.iter = (int)(it & 0x3fffffff);
            if (node ? bp_launch_node_iteration(d->dv, d->dc, p, q == 0, st) : bp_launch_stream_iteration(d->dv, d->dc, p, q == 0, st))
                return fail(SCLDPC_EINVAL, "unsupported degrees");
        }
        const int slot = nchunk & 1;
        p.harvest_parity = slot;
        p.iter = (int)(it & 0x3fffffff);         // the iteration that runs next (its parity names the planes)
        if (adaptive) CU(cudaMemsetAsync(p.alive_total + 1 + slot, 0x7f, sizeof(int), st));
        if (node) bp_launch_node_settle(d->dv, d->dc, p, st);
        bp_launch_count_pairs(d->dv, d->dc, p, st);
        bp_launch_stream_harvest(p, (cfg->flags & SCLDPC_F_EXP_ALL) ? 1 : 0, st);
        if (node) {
            bp_launch_node_arm(p, st);
            bp_launch_node_compact(p, st);
        }
        bp_launch_node_alive_list(p, slot, st);
        CU_LAUNCHES();
        CU(cudaMemcpyAsync(hf + 8 * slot, p.alive_total, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(ev[slot], st));
        pending[slot] = true;
        nchunk++;
        const int prev = nchunk & 1;
        if (pending[prev]) {
            CU(cudaEventSynchronize(ev[prev]));
            pending[prev] = false;
            if (hf[8 * prev] == 0) break;
            // grids of the next chunk: the graphs that were alive at that harvest
            p.glist = p.glist2 + (size_t)prev * p.G;
            p.n_glist = hf[8 * prev + 6 + prev];
            if (p.n_glist < 1 || p.n_glist > p.G) { p.glist = nullptr; p.n_glist = 0; }
            const int mean_it = hf[8 * prev + 1 + prev];   // 0x7f7f7f7f: no graph still decoding has harvested a frame yet
            if (adaptive && mean_it != 0x7f7f7f7f && mean_it > 0) {
                H = (int)(sqrt(0.1 * HARVEST_C10 * mean_it) + 0.5);
                H = H < 8 ? 8 : (H > 64 ? 64 : H);
            }
        }
    }
    if (iters_launched_host) *iters_launched_host = it;
    return 0;
}

// Full BP (unlimited iterations) over a stream of cfg->frames_per_graph frames per graph with lane recycling.
extern "C" int scldpc_bp_stream(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg,
                                const scldpc_stream_out_t *out, void *workspace_dev, size_t workspace_bytes,
                                long long *iters_launched_host, void *stream)
{
    return bp_stream_impl(d, b, cfg, nullptr, 0, out, workspace_dev, workspace_bytes, iters_launched_host, stream);
}

// The same stream with checkpoints at the caps of an ascending list (include/scldpc.h).
extern "C" int scldpc_bp_stream_caps(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg,
                                     const int32_t *caps_host, int n_caps, const scldpc_stream_caps_out_t *out,
                                     void *workspace_dev, size_t workspace_bytes, long long *iters_launched_host, void *stream)
{
    if (n_caps < 1 || n_caps > SCLDPC_MAX_CAPS) return fail(SCLDPC_EINVAL, "n_caps must be in [1, %d], got %d", SCLDPC_MAX_CAPS, n_caps);
    if (!caps_host) return fail(SCLDPC_EINVAL, "caps_host is NULL");
    for (int k = 0; k < n_caps; k++) {
        const bool unlimited_last = k == n_caps - 1 && caps_host[k] <= 0;
        if (!unlimited_last && caps_host[k] < 1) return fail(SCLDPC_EINVAL, "cap %d is %d: caps must be >= 1 (only the last may be <= 0, unlimited)", k, caps_host[k]);
        if (k > 0 && !unlimited_last && caps_host[k] <= caps_host[k - 1])
            return fail(SCLDPC_EINVAL, "caps must be strictly ascending: cap %d (%d) <= cap %d (%d)", k, caps_host[k], k - 1, caps_host[k - 1]);
    }
    if (!cfg) return fail(SCLDPC_EINVAL, "bad stream configuration");
    if (cfg->max_it != 0) return fail(SCLDPC_EINVAL, "cfg->max_it must be 0 with caps: the caps replace it");
    if (cfg->flags & SCLDPC_F_MESSAGES) return fail(SCLDPC_EINVAL, "frame streams with caps need the node-state sweeps (no SCLDPC_F_MESSAGES)");
    if (!out) return fail(SCLDPC_EINVAL, "output pointer is NULL");
    const scldpc_stream_out_t o{out->iters_dev, out->residual_dev, out->blocks_err_dev, out->erasures_exp_dev, out->blocks_err_exp_dev};
    return bp_stream_impl(d, b, cfg, caps_host, n_caps, &o, workspace_dev, workspace_bytes, iters_launched_host, stream);
}

// first_window / n_windows: the windows [first_window, first_window + n_windows) of the chain (n_windows < 0: to the end).
// pending_dev (node-state sweeps only): caller-owned second plane [G][n][W]; with resume != 0 the call continues from the
// state the caller left in out->erased_dev (what the CNs see) and pending_dev (what each VN has been told so far) instead
// of initialising both from the channel -- the streaming decoder carries them from one piece of the chain to the next.
static int bp_window_impl(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                          int first_window, int n_windows, uint64_t *pending_dev, int resume,
                          const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                          int64_t *edge_updates_host, void *stream);

extern "C" int scldpc_bp_window(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                                const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                                int64_t *edge_updates_host, void *stream)
{
    return bp_window_impl(d, b, W, max_it, init_it, flags, 0, -1, nullptr, 0, out, workspace_dev, workspace_bytes, edge_updates_host, stream);
}

extern "C" int scldpc_bp_window_range(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                                      int first_window, int n_windows, uint64_t *pending_dev, int resume,
                                      const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                                      int64_t *edge_updates_host, void *stream)
{
    if (flags & SCLDPC_F_MESSAGES) return fail(SCLDPC_EINVAL, "window ranges need the node-state sweeps (no SCLDPC_F_MESSAGES)");
    if (!pending_dev) return fail(SCLDPC_EINVAL, "pending_dev is NULL");
    if (first_window < 0) return fail(SCLDPC_EINVAL, "first_window must be >= 0");
    if (d && d->n_frames < 1) return fail(SCLDPC_EINVAL, "n_frames must be >= 1");
    return bp_window_impl(d, b, W, max_it, init_it, flags, first_window, n_windows, pending_dev, resume, out, workspace_dev,
                          workspace_bytes, edge_updates_host, stream);
}

static int bp_window_impl(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                          int first_window, int n_windows, uint64_t *pending_dev, int resume,
                          const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                          int64_t *edge_updates_host, void *stream)
{
    if (flags & SCLDPC_F_TRAJECTORY) return fail(SCLDPC_EINVAL, "the window decoder records no trajectory");
    if (W < 1) return fail(SCLDPC_EINVAL, "W must be >= 1");
    BpParams p;
    int rc = setup_params(d, b, flags, out, workspace_dev, workspace_bytes, &p);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool term = flags & SCLDPC_F_TERMINATED, square = flags & SCLDPC_F_SQUARE;
    const int cap = max_it <= 0 ? INT_MAX : max_it;
    const int cap0 = init_it <= 0 ? cap : init_it;                 // BP_SW.c:2099-2102
    const int ms = d->dv - 1, L = d->L, vp = d->vns_pos, cp = d->cns_pos;
    const int nwin = square ? L : L + ms;                          // BP_SW.c:672 / BP_FULL.c:668
    const int cn_clip = term ? p.nk : L * cp;
    // SCLDPC_F_MESSAGES selects the message-passing sweeps (the implementation of record); the default is their node-state
    // form (bpw_*_node_kernel in bp_kernels.cu): same decisions, counters and per-window stopping, about a third of the traffic
    const bool node = !(flags & SCLDPC_F_MESSAGES) && d->n_frames > 0;
    if (node) {
        p.xb = pending_dev ? reinterpret_cast<u128 *>(pending_dev) : p.y;   // the wave-tracking plane is free in window mode
        // resolution lists pay when few rows change per iteration, i.e. when the window is long against the wave (about 10
        // positions); short windows copy the VN window instead (bp_window_node_kernels.cu)
        p.win_lists = (long long)(W + ms) * 2 >= L ? 1 : 0;
        bp_launch_init_ctrl_only(p, d->n_frames, st);
        bp_launch_window_node_init(p, st, resume != 0);
    } else {
        bp_launch_init(p, d->dv, d->dc, 0, d->n_frames, st);
        CU(cudaMemsetAsync(out->erased_dev, 0, sizeof(u64) * (size_t)p.G * p.n * p.W, st));
    }
    CU(cudaGetLastError());
    const int win_end = (n_windows < 0 || first_window + (long long)n_windows > nwin) ? nwin : first_window + n_windows;
    for (int posW = first_window; posW < win_end && d->n_frames > 0; posW++) {
        long long c0 = (long long)posW * cp, c1 = c0 + (long long)W * cp;
        if (c1 > cn_clip) c1 = cn_clip;
        if (c1 < c0) c1 = c0;
        long long v0, v1;
        if (square) { v0 = (long long)posW * vp; v1 = v0 + (long long)W * vp; }
        else if (posW <= ms) { v0 = 0; v1 = (long long)(W + posW) * vp; }
        else { v0 = (long long)(posW - ms) * vp; v1 = v0 + (long long)(W + ms) * vp; }
        if (v1 > p.n) v1 = p.n;
        p.c0 = (int)c0; p.c1 = (int)c1; p.v0 = (int)v0; p.v1 = (int)v1;
        p.stall_at_first = (v1 - v0 == p.n);
        // edge updates of one iteration: CN position q carries vns_pos edges from each VN position q-i in [0,L)
        long long ce = 0;
        for (long long q = c0 / cp; q < c1 / cp; q++)
            for (int i = 0; i < d->dv; i++)
                if (q - i >= 0 && q - i < L) ce += vp;
        p.win_edges = ce + (v1 - v0) * d->dv;
        bp_launch_window_begin(p, d->n_frames, st);
        const int NumIt = (square && posW == 0) ? cap0 : cap;      // BP_SW.c:699-702
        if ((rc = run_iterations(&p, d->dv, d->dc, NumIt, false, true, false, st, nullptr, node))) return rc;
        if (node && bp_launch_window_node_end(d->dv, d->dc, p, st)) return fail(SCLDPC_EINVAL, "unsupported degrees");
    }
    BpFinalOut fo{out->residual_dev, out->blocks_err_dev, out->erasures_exp_dev, out->blocks_err_exp_dev, out->erasures_p1_dev,
                  1, square ? ms : 0, square ? W - 2 : W - 2 - ms};   // posW in [ms, W-2] (BP_SW.c:846-847)
    bp_launch_finalize(d->dv, d->dc, p, fo, st);
    CU(cudaGetLastError());
    if (edge_updates_host) {
        std::vector<long long> w((size_t)p.G * p.lanes);
        CU(cudaMemcpyAsync(w.data(), p.work, sizeof(long long) * w.size(), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        long long tot = 0;
        for (long long x : w) tot += x;
        *edge_updates_host = tot;
    }
    return 0;
}

// ---- peeling decoder ------------------------------------------------------------------------------------------------
extern "C" void scldpc_philox_picks(uint64_t seed, uint64_t frame_id, int n, uint32_t *out_host)
{
    if (out_host && n > 0) peel_picks_host(seed, frame_id, n, out_host);
}

extern "C" size_t scldpc_peel_workspace_bytes(const scldpc_dims_t *d, int n_cn_all, int total_size)
{
    if (check_dims(d) || have_device()) return 0;
    const int grid = peel_grid(total_size, (long long)d->n_graphs * d->n_frames, n_cn_all);
    if (grid < 0) { fail(SCLDPC_EINVAL, "total_size too large for the shared-memory bitmap"); return 0; }
    return sizeof(u64) * ((size_t)grid * peel_state_words(n_cn_all, total_size) + 1);     // + the frame counter
}

extern "C" int scldpc_peel_trajectories(const scldpc_dims_t *d, const int32_t *vn_cn_dev, const uint64_t *chan_dev, int n_cn_all,
                                        int total_size, int num_steps, uint64_t seed, uint64_t first_frame_id, int32_t *r1_dev,
                                        int32_t *recovered_dev, int32_t *n_erased_dev, void *workspace_dev, size_t workspace_bytes,
                                        void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!vn_cn_dev || !chan_dev || !recovered_dev || !n_erased_dev || !workspace_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if (total_size < 1 || total_size > n_cn_all || num_steps < 0) return fail(SCLDPC_EINVAL, "bad total_size / num_steps");
    if ((rc = have_device())) return rc;
    const long long frames = (long long)d->n_graphs * d->n_frames;
    if (frames == 0) return 0;
    const int grid = peel_grid(total_size, frames, n_cn_all);
    if (grid < 0) return fail(SCLDPC_EINVAL, "total_size too large for the shared-memory bitmap");
    const size_t st_words = (size_t)grid * peel_state_words(n_cn_all, total_size);
    if (workspace_bytes < sizeof(u64) * (st_words + 1)) return fail(SCLDPC_ENOMEM, "workspace too small");
    PeelParams p;
    memset(&p, 0, sizeof p);
    p.n = d->L * d->vns_pos; p.dv = d->dv; p.n_cn_all = n_cn_all; p.total_size = total_size; p.num_steps = num_steps;
    p.W = d->n_words; p.n_frames = d->n_frames; p.G = d->n_graphs;
    p.vn_cn = vn_cn_dev; p.chan = reinterpret_cast<const u64 *>(chan_dev); p.state = static_cast<u64 *>(workspace_dev);
    p.r1 = r1_dev; p.recovered = recovered_dev; p.n_erased = n_erased_dev; p.seed = seed; p.first_frame = first_frame_id;
    p.next = p.state + st_words;                 // frames are handed out dynamically once every warp has its first one
    CU(cudaMemsetAsync(p.next, 0, sizeof(u64), static_cast<cudaStream_t>(stream)));
    if (peel_launch(p, grid, static_cast<cudaStream_t>(stream))) return fail(SCLDPC_EINVAL, "peeling launch configuration failed");
    CU(cudaGetLastError());
    return 0;
}

extern "C" int scldpc_peel_variance_accumulate(const int32_t *r1_dev, int n_frames, int row_len, const double *theory_dev, int S,
                                               double M, double *ssq_dev, int64_t *counts_dev, void *stream)
{
    if (!r1_dev || !theory_dev || !ssq_dev || !counts_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if (S < 0 || S > row_len || n_frames < 0) return fail(SCLDPC_EINVAL, "bad sizes");
    int rc = have_device();
    if (rc) return rc;
    if (S == 0) return 0;
    peel_variance_launch(r1_dev, n_frames, row_len, theory_dev, S, M, ssq_dev, reinterpret_cast<long long *>(counts_dev),
                         static_cast<cudaStream_t>(stream));
    CU(cudaGetLastError());
    return 0;
}

// Per-position results of the last scldpc_bp_full / scldpc_bp_window call on this workspace (device to device):
// pos_cnt[g][p][lane] = erased VNs of position p, pos_pairs[g][p][lane] = accepted size-two stopping sets of position p
// (get_deg_two_ss, BP_FULL.c:1227: the expurgated count of a position is pos_cnt - 2*pos_pairs).
extern "C" int scldpc_bp_position_counts(const scldpc_dims_t *d, uint32_t flags, void *workspace_dev, int32_t *pos_cnt_dev,
                                         int32_t *pos_pairs_dev, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!workspace_dev || !pos_cnt_dev || !pos_pairs_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    BpParams p;
    carve(d, flags, workspace_dev, &p);
    const size_t bytes = sizeof(int32_t) * (size_t)d->n_graphs * d->L * 64 * d->n_words;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CU(cudaMemcpyAsync(pos_cnt_dev, p.pos_cnt, bytes, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(pos_pairs_dev, p.pos_pairs, bytes, cudaMemcpyDeviceToDevice, st));
    return 0;
}

// ---- pairwise-complete moments behind DataFrame.corr() in calc_theta_explicit_ss_bounds (EST.py:161-189) ----
extern "C" int scldpc_pairwise_moments_accumulate(const int32_t *r1_dev, int n_frames, int row_len, int start, int step, int K,
                                                  int64_t *acc_dev, void *stream)
{
    if (!r1_dev || !acc_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if (n_frames < 0 || K < 1 || step < 1 || start < 0 || start + (long long)(K - 1) * step >= row_len)
        return fail(SCLDPC_EINVAL, "sampled columns out of range");
    int rc = have_device();
    if (rc) return rc;
    if (n_frames == 0) return 0;
    corr_moments_launch(r1_dev, n_frames, row_len, start, step, K, reinterpret_cast<long long *>(acc_dev), static_cast<cudaStream_t>(stream));
    CU(cudaGetLastError());
    return 0;
}

// ---- per-iteration moments of BP trajectories (the notebook's nu_BP / mean dVNs inputs, NB cells 40-42) ----
extern "C" int scldpc_bp_trajectory_moments(const scldpc_dims_t *d, const int32_t *rows_dev, const int32_t *iters_dev, int max_rows,
                                            int64_t *acc_dev, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!rows_dev || !iters_dev || !acc_dev || max_rows < 1) return fail(SCLDPC_EINVAL, "NULL pointer or max_rows < 1");
    if ((rc = have_device())) return rc;
    traj_moments_launch(rows_dev, iters_dev, d->n_graphs, max_rows, 64 * d->n_words, d->n_frames, reinterpret_cast<long long *>(acc_dev),
                        static_cast<cudaStream_t>(stream));
    CU(cudaGetLastError());
    return 0;
}

// ---- stopping sets of the residual graph (simulate_sc_ldpc, PD.py:659-691 + extract_stopping_sets PD.py:1077-1095) ----
extern "C" int scldpc_bp_stopping_sets(const scldpc_dims_t *d, const scldpc_batch_t *b, const uint64_t *erased_dev,
                                       const uint8_t *counted_pos_host, int32_t *out_dev, void *stream)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!degrees_supported(d->dv, d->dc)) return fail(SCLDPC_EINVAL, "(dv,dc)=(%d,%d) not instantiated", d->dv, d->dc);
    if (!b || !b->vn_cn_dev || !b->cn_edge_dev || !erased_dev || !out_dev) return fail(SCLDPC_EINVAL, "NULL pointer");
    if ((rc = have_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SsParams p;
    memset(&p, 0, sizeof p);
    p.dv = d->dv; p.dc = d->dc; p.n = d->L * d->vns_pos; p.nk = (d->L + d->dv - 1) * d->cns_pos; p.E = p.n * d->dv;
    p.L = d->L; p.vns_pos = d->vns_pos; p.G = d->n_graphs; p.W = d->n_words; p.chunks = d->n_words / 2; p.lanes = 64 * d->n_words;
    while ((1 << p.chunk_shift) < p.chunks) p.chunk_shift++;
    p.vn_cn = b->vn_cn_dev; p.cn_edge = b->cn_edge_dev; p.x = reinterpret_cast<const u128 *>(erased_dev); p.out = out_dev;
    const size_t cnt_bytes = sizeof(int) * (size_t)p.G * p.L * p.lanes, ge3_bytes = sizeof(u128) * (size_t)p.G * p.nk * p.chunks;
    char *scratch = nullptr;
    const size_t cnt_al = align_up(cnt_bytes), L_al = align_up((size_t)d->L);
    CU(cudaMallocAsync(&scratch, 2 * cnt_al + ge3_bytes + L_al, st));
    p.pos_lost = reinterpret_cast<int *>(scratch);
    p.pos_big = reinterpret_cast<int *>(scratch + cnt_al);
    p.ge3 = reinterpret_cast<u128 *>(scratch + 2 * cnt_al);
    unsigned char *counted = reinterpret_cast<unsigned char *>(scratch + 2 * cnt_al + ge3_bytes);
    p.counted = counted;
    CU(cudaMemsetAsync(scratch, 0, 2 * cnt_al, st));
    std::vector<unsigned char> cp(d->L, 1);
    if (counted_pos_host) cp.assign(counted_pos_host, counted_pos_host + d->L);
    CU(cudaMemcpyAsync(counted, cp.data(), d->L, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));               // cp leaves scope
    if (ss_launch(p, st)) return fail(SCLDPC_EINVAL, "unsupported degrees");
    CU_LAUNCHES();
    CU(cudaFreeAsync(scratch, st));
    return 0;
}

// ---- multi-GPU: the only collective of the path ------------------------------------------------------------------------
// Sum of an int64 counter / accumulator vector over the ranks of a caller-owned NCCL communicator (the reference merges its
// per-process files offline with awk / pickle sums, NB:565, NB:1195, notebook cell 23).  NCCL is resolved at call time with
// dlopen, so the library has no link-time dependency on it and uses the NCCL the calling process has already loaded.
#include <dlfcn.h>
extern "C" int scldpc_allreduce_counters(void *nccl_comm, int64_t *counters_dev, int n_int64, void *stream)
{
    if (!nccl_comm || !counters_dev || n_int64 < 0) return fail(SCLDPC_EINVAL, "NULL communicator / buffer");
    if (n_int64 == 0) return 0;
    typedef int (*allreduce_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
    static allreduce_fn fn = nullptr;
    if (!fn) {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return fail(SCLDPC_ECUDA, "NCCL not found: %s", dlerror());
        fn = reinterpret_cast<allreduce_fn>(dlsym(h, "ncclAllReduce"));
        if (!fn) return fail(SCLDPC_ECUDA, "ncclAllReduce not found in libnccl");
    }
    const int nccl_int64 = 4, nccl_sum = 0;      // ncclDataType_t / ncclRedOp_t values of nccl.h (stable ABI)
    const int rc = fn(counters_dev, counters_dev, (size_t)n_int64, nccl_int64, nccl_sum, nccl_comm, static_cast<cudaStream_t>(stream));
    if (rc != 0) return fail(SCLDPC_ECUDA, "ncclAllReduce failed with ncclResult_t %d", rc);
    return 0;
}

// ---- instrumentation --------------------------------------------------------------------------------------------
// Positions swept by the last scldpc_bp_full call on this workspace, summed over graphs and iterations:
// out[0] = CN positions, out[1] = VN positions (a sweep of everything would be iterations*(L+dv-1) and iterations*L).
extern "C" int scldpc_bp_sweep_stats(const scldpc_dims_t *d, uint32_t flags, void *workspace_dev, long long *out_host)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!workspace_dev || !out_host) return fail(SCLDPC_EINVAL, "NULL pointer");
    BpParams p;
    carve(d, flags, workspace_dev, &p);
    std::vector<long long> h(2 * (size_t)d->n_graphs);
    CU(cudaMemcpy(h.data(), p.swept, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    out_host[0] = out_host[1] = 0;
    for (int g = 0; g < d->n_graphs; g++) { out_host[0] += h[2 * g]; out_host[1] += h[2 * g + 1]; }
    return 0;
}

extern "C" long long scldpc_launch_count(int reset)
{
    long long v = g_prof.launches;
    if (reset) g_prof.launches = 0;
    return v;
}

// Times the CN and VN sweeps of every sample_every-th iteration with CUDA events on the launching stream.
extern "C" int scldpc_profile_begin(int sample_every, int max_samples)
{
    int rc = have_device();
    if (rc) return rc;
    if (sample_every < 1 || max_samples < 1) return fail(SCLDPC_EINVAL, "sample_every and max_samples must be >= 1");
    if (g_prof.ev) {
        for (int i = 0; i < 3 * g_prof.max_samples; i++) cudaEventDestroy(g_prof.ev[i]);
        delete[] g_prof.ev;
        delete[] g_prof.iter_idx;
    }
    g_prof.ev = new cudaEvent_t[3 * (size_t)max_samples];
    g_prof.iter_idx = new int[max_samples];
    for (int i = 0; i < 3 * max_samples; i++) CU(cudaEventCreate(&g_prof.ev[i]));
    g_prof.max_samples = max_samples;
    g_prof.n_samples = 0;
    g_prof.sample_every = sample_every;
    return 0;
}

// Stops sampling; returns the number of samples and, per sample, the iteration index and the two durations (ms).
extern "C" int scldpc_profile_end(int *n_samples, int *iter_idx, float *cn_ms, float *vn_ms, int capacity)
{
    g_prof.sample_every = 0;
    if (!n_samples) return fail(SCLDPC_EINVAL, "n_samples is NULL");
    CU(cudaDeviceSynchronize());
    int m = g_prof.n_samples < capacity ? g_prof.n_samples : capacity;
    for (int i = 0; i < m; i++) {
        if (iter_idx) iter_idx[i] = g_prof.iter_idx[i];
        float a = 0, b = 0;
        CU(cudaEventElapsedTime(&a, g_prof.ev[3 * i], g_prof.ev[3 * i + 1]));
        CU(cudaEventElapsedTime(&b, g_prof.ev[3 * i + 1], g_prof.ev[3 * i + 2]));
        if (cn_ms) cn_ms[i] = a;
        if (vn_ms) vn_ms[i] = b;
    }
    *n_samples = m;
    g_prof.n_samples = 0;
    return 0;
}

// ---- host-buffer convenience entry point --------------------------------------------------------------------------

// Stream-ordered allocations from the device's default pool; the pool keeps freed memory (release threshold raised
// once), so repeated calls do not pay cudaMalloc / cudaFree.
struct DevBuf {
    void *p = nullptr;
    cudaStream_t st = nullptr;
    ~DevBuf() { if (p) cudaFreeAsync(p, st); }
    int alloc(size_t bytes, cudaStream_t s = nullptr) { st = s; return cudaMallocAsync(&p, bytes ? bytes : 1, s) == cudaSuccess ? 0 : -1; }
};

// The host-buffer entry points work on a stream of the calling host thread, so that calls from different host threads overlap
// on the device (two batches in flight hide the tail of one batch's frame streams behind the next batch, bench.py).
static cudaStream_t host_call_stream()
{
    static thread_local cudaStream_t s = nullptr;
    if (!s && cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) s = nullptr;
    return s;
}

static void keep_pool_memory()
{
    static bool done = false;
    if (done) return;
    done = true;
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
}

// Host-buffer form of scldpc_bp_stream: graph tables come from host memory, per-frame results return to host memory
// (int32 [G][frames_per_graph] each); the channel realisations are drawn on the device.
extern "C" int scldpc_stream_host(const scldpc_dims_t *d, const int32_t *vn_cn_host, const scldpc_stream_cfg_t *cfg,
                                  int32_t *iters_host, int32_t *residual_host, int32_t *blocks_err_host,
                                  int32_t *erasures_exp_host, int32_t *blocks_err_exp_host, long long *iters_launched_host)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!vn_cn_host || !cfg) return fail(SCLDPC_EINVAL, "NULL input pointer");
    if ((rc = have_device())) return rc;
    keep_pool_memory();
    const size_t G = d->n_graphs, B = cfg->frames_per_graph > 0 ? cfg->frames_per_graph : 0;
    const size_t n = (size_t)d->L * d->vns_pos, nk = (size_t)(d->L + d->dv - 1) * d->cns_pos, E = n * d->dv;
    DevBuf vn_cn, vn_slot, cn_edge, scratch, ws, res;
    const size_t ws_bytes = scldpc_bp_stream_workspace_bytes(d, cfg->flags);
    cudaStream_t st = host_call_stream();
    if (vn_cn.alloc(4 * G * E, st) || vn_slot.alloc(4 * G * E, st) || cn_edge.alloc(4 * G * nk * d->dc, st) || scratch.alloc(4 * G * nk, st) ||
        ws.alloc(ws_bytes, st) || res.alloc(4 * 5 * G * B, st))
        return fail(SCLDPC_ECUDA, "cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaMemcpyAsync(vn_cn.p, vn_cn_host, 4 * G * E, cudaMemcpyHostToDevice, st));
    scldpc_batch_t b{static_cast<int32_t *>(vn_cn.p), static_cast<int32_t *>(vn_slot.p), static_cast<int32_t *>(cn_edge.p), nullptr};
    if ((rc = scldpc_graph_build_tables(d, &b, static_cast<int32_t *>(scratch.p), st))) return rc;
    int32_t *r = static_cast<int32_t *>(res.p);
    CU(cudaMemsetAsync(r, 0, 4 * 5 * G * B, st));
    scldpc_stream_out_t out{r, r + G * B, r + 2 * G * B, r + 3 * G * B, r + 4 * G * B};
    if ((rc = scldpc_bp_stream(d, &b, cfg, &out, ws.p, ws_bytes, iters_launched_host, st))) return rc;
    int32_t *dsts[5] = {iters_host, residual_host, blocks_err_host, erasures_exp_host, blocks_err_exp_host};
    for (int a = 0; a < 5; a++)
        if (dsts[a]) CU(cudaMemcpyAsync(dsts[a], r + a * G * B, 4 * G * B, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int scldpc_decode_host(const scldpc_dims_t *d, const int32_t *vn_cn_host, const uint8_t *erased_host, int W, int max_it,
                                  int init_it, uint32_t flags, int32_t *iters_host, int32_t *residual_host,
                                  int32_t *blocks_err_host, int32_t *erasures_exp_host, int32_t *blocks_err_exp_host,
                                  int32_t *erasures_p1_host, uint8_t *vn_erased_host, int32_t *rows_host, int max_rows)
{
    int rc = check_dims(d);
    if (rc) return rc;
    if (!vn_cn_host || !erased_host) return fail(SCLDPC_EINVAL, "NULL input pointer");
    if ((rc = have_device())) return rc;
    const size_t G = d->n_graphs, Wd = d->n_words, lanes = 64 * Wd, F = d->n_frames;
    const size_t n = (size_t)d->L * d->vns_pos, nk = (size_t)(d->L + d->dv - 1) * d->cns_pos, E = n * d->dv;
    const bool traj = (flags & SCLDPC_F_TRAJECTORY) && W == 0;
    if ((flags & SCLDPC_F_TRAJECTORY) && (!rows_host || max_rows <= 0)) return fail(SCLDPC_EINVAL, "rows_host / max_rows missing");
    keep_pool_memory();
    DevBuf vn_cn, vn_slot, cn_edge, chan, scratch, ws, res, xbuf, rows, bytes;
    const uint32_t kflags = flags & ~SCLDPC_F_CHAN_PACKED;
    const size_t ws_bytes = scldpc_bp_workspace_bytes(d, kflags);
    if (vn_cn.alloc(4 * G * E) || vn_slot.alloc(4 * G * E) || cn_edge.alloc(4 * G * nk * d->dc) || chan.alloc(8 * G * n * Wd) ||
        scratch.alloc(4 * G * nk) || ws.alloc(ws_bytes) || res.alloc(4 * 6 * G * lanes) || xbuf.alloc(8 * G * n * Wd) ||
        (traj && rows.alloc(4 * 3 * G * (size_t)max_rows * lanes)) || (vn_erased_host && bytes.alloc(G * F * n)))
        return fail(SCLDPC_ECUDA, "cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaStream_t st = nullptr;
    CU(cudaMemcpyAsync(vn_cn.p, vn_cn_host, 4 * G * E, cudaMemcpyHostToDevice, st));
    scldpc_batch_t b{static_cast<int32_t *>(vn_cn.p), static_cast<int32_t *>(vn_slot.p), static_cast<int32_t *>(cn_edge.p),
                     static_cast<uint64_t *>(chan.p)};
    if ((rc = scldpc_graph_build_tables(d, &b, static_cast<int32_t *>(scratch.p), st))) return rc;
    if (flags & SCLDPC_F_CHAN_PACKED) CU(cudaMemcpyAsync(chan.p, erased_host, 8 * G * n * Wd, cudaMemcpyHostToDevice, st));
    else if ((rc = scldpc_channel_pack_host(d, erased_host, static_cast<uint64_t *>(chan.p), st))) return rc;
    int32_t *r = static_cast<int32_t *>(res.p);
    scldpc_bp_out_t out{r, r + G * lanes, r + 2 * G * lanes, r + 3 * G * lanes, r + 4 * G * lanes, r + 5 * G * lanes,
                        static_cast<uint64_t *>(xbuf.p), traj ? static_cast<int32_t *>(rows.p) : nullptr, traj ? max_rows : 0};
    if (traj) CU(cudaMemsetAsync(rows.p, 0, 4 * 3 * G * (size_t)max_rows * lanes, st));
    if (W == 0) rc = scldpc_bp_full(d, &b, max_it, kflags, 0, &out, ws.p, ws_bytes, nullptr, st);
    else rc = scldpc_bp_window(d, &b, W, max_it, init_it, kflags & ~SCLDPC_F_TRAJECTORY, &out, ws.p, ws_bytes, nullptr, st);
    if (rc) return rc;
    std::vector<int32_t> h(6 * G * lanes);
    CU(cudaMemcpyAsync(h.data(), r, 4 * h.size(), cudaMemcpyDeviceToHost, st));
    if (vn_erased_host) {
        bits_unpack(static_cast<u64 *>(xbuf.p), static_cast<uint8_t *>(bytes.p), (int)G, (int)n, (int)Wd, (int)F, st);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(vn_erased_host, bytes.p, G * F * n, cudaMemcpyDeviceToHost, st));
    }
    std::vector<int32_t> hr;
    if (traj) {
        hr.resize(3 * G * (size_t)max_rows * lanes);
        CU(cudaMemcpyAsync(hr.data(), rows.p, 4 * hr.size(), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    int32_t *dsts[6] = {iters_host, residual_host, blocks_err_host, erasures_exp_host, blocks_err_exp_host, erasures_p1_host};
    for (int a = 0; a < 6; a++)
        if (dsts[a])
            for (size_t g = 0; g < G; g++)
                memcpy(dsts[a] + g * F, h.data() + (a * G + g) * lanes, 4 * F);
    if (traj)   // [G][max_rows][lanes][3] -> [G][n_frames][max_rows][3]
        for (size_t g = 0; g < G; g++)
            for (size_t f = 0; f < F; f++)
                for (int t = 0; t < max_rows; t++)
                    memcpy(rows_host + ((g * F + f) * max_rows + t) * 3, hr.data() + ((g * max_rows + t) * lanes + f) * 3, 12);
    return 0;
}
