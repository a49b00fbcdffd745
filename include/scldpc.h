/*
 * scldpc.h -- C ABI of libscldpc.so, the B200 (sm_100a) Monte-Carlo decoding engine for (dv,dc)-regular
 * SC-LDPC codes over the BEC.
 *
 * The reference (rsokolovskii/fl_scaling_sc_ldpc) has no FFI of its own: its hot path is reached through C
 * functions operating on file-scope tables and through Python callables.  Each entry point below names the
 * reference interface it replaces (file:line; abbreviations as in SURVEY.md):
 *   BP_FULL.c = simulators_sc_ldpc/bp_decoding/SC_LDPC_Simulator_BPDecoder_BEC_full_BP_LimIter_OlmosRandomEnsemble.c
 *   BP_SW.c   = simulators_sc_ldpc/bp_decoding/SC_LDPC_Simulator_BPDecoder_BEC_SlidingWindow_LimIter_OlmosRandomEnsemble.c
 *   BP_TRAJ.c = simulators_sc_ldpc/bp_decoding/trajectories_SC_LDPC_Simulator_BPDecoder_BEC_full_BP_OlmosRandomEnsemble.c
 *   PD.py     = simulators_sc_ldpc/peeling_decoding/peeling_decoding.py
 *   SC.py     = simulators_sc_ldpc/peeling_decoding/sc_ldpc.py
 *
 * Conventions
 *  - Plain C types only.  Pointers named *_dev are device pointers (owned by the caller, e.g. a torch
 *    tensor's data_ptr()); pointers named *_host are host pointers.  `stream` is a cudaStream_t passed as
 *    void* (NULL = default stream).  Every function returns 0 on success and a negative SCLDPC_E* code on
 *    failure; scldpc_last_error() returns a thread-local message.  There is NO CPU fallback: without a CUDA
 *    device every compute entry point fails with SCLDPC_ECUDA.
 *  - Host threads may call concurrently on different streams / workspaces: all library state is per calling thread.
 *    The *_host entry points (host buffers in, host buffers out) work on a stream owned by the calling thread.
 *  - A batch holds n_graphs independent graph realisations; each graph decodes 64*n_words frames at once,
 *    bit-sliced: bit b of 64-bit word w of a node is that node's value in frame 64*w+b of the graph.
 *    n_words must be a power of two in [2,16].
 *  - M := vns_pos = VNs per position (paper / Python convention); the C files' Def_M equals cns_pos.
 *    n = L*vns_pos VNs, nk = (L+dv-1)*cns_pos CNs, E = n*dv edges per graph.
 */
#ifndef SCLDPC_H
#define SCLDPC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCLDPC_OK 0
#define SCLDPC_EINVAL (-1)   /* bad argument                       */
#define SCLDPC_ECUDA (-2)    /* CUDA runtime error / no device     */
#define SCLDPC_ENOMEM (-3)   /* workspace too small                */
#define SCLDPC_EGRAPH (-4)   /* malformed graph (CN degree > dc..) */

/* decoder flags */
#define SCLDPC_F_TERMINATED 1u   /* is_term (BP_TRAJ.c:901): 0 = truncated, tail CNs always send erasures      */
#define SCLDPC_F_TRAJECTORY 2u   /* record (deg_1_iter, dVNs, first erased position) per iteration (node-state sweep with a CN
                                    latch and per-position counters, or the message kernels with SCLDPC_F_MESSAGES)          */
#define SCLDPC_F_SQUARE 4u       /* window decoder: square window (BP_SW.c) instead of classical (BP_FULL.c)    */
#define SCLDPC_F_EXP_ALL 8u      /* expurgated statistics over all positions (decodeBP_SW) instead of the first */
#define SCLDPC_F_STREAM 32u      /* internal: workspace sizing of scldpc_bp_stream */
#define SCLDPC_F_CHAN_PACKED 16u /* scldpc_decode_host: erased_host is already bit-sliced, uint64 [G][n][n_words] */
#define SCLDPC_F_MESSAGES 64u    /* pass explicit Lji / Lij messages (the implementation of record) instead of the node-state
                                    sweeps, which yield the same erased set at every iteration (DESIGN.md section 4).  Applies
                                    to scldpc_bp_full without a trajectory, scldpc_bp_window and scldpc_bp_stream; workspace
                                    sizes depend on it, so pass the same flags to the *_workspace_bytes query and the call  */
#define SCLDPC_F_NODE_TRAJ 256u  /* scldpc_bp_full with SCLDPC_F_TRAJECTORY: node-state sweep even above 32768 VNs per position   */
#define SCLDPC_F_NO_WAVE 128u    /* scldpc_bp_full with messages: sweep every position in every iteration (testing)          */

typedef struct {
    int32_t dv, dc;        /* variable / check node degree (Def_dv, Def_dc; BP_FULL.c:22-23)                */
    int32_t L;             /* chain length (Def_L)                                                          */
    int32_t vns_pos;       /* VNs per position (Def_VNsPos = M)                                             */
    int32_t cns_pos;       /* CNs per position (Def_CNsPos = Def_M); vns_pos*dv must equal cns_pos*dc       */
    int32_t n_graphs;      /* graph realisations in the batch                                               */
    int32_t n_words;       /* 64-bit lane words per node; frames per graph = 64*n_words                     */
    int32_t n_frames;      /* valid frames per graph (<= 64*n_words); remaining lanes are ignored           */
} scldpc_dims_t;

/* Device buffers of a batch.  Sizes in elements, G = n_graphs, W = n_words, n/nk/E per graph as above. */
typedef struct {
    const int32_t *vn_cn_dev;   /* [G][n][dv]   CN index of edge i of VN v (VNdegree[v][1+i], BP_FULL.c:87)    */
    int32_t *vn_slot_dev;       /* [G][n][dv]   c*dc+j: slot of that edge in its CN row (built by the library) */
    int32_t *cn_edge_dev;       /* [G][nk][dc]  v*dv+i of the j-th edge of CN c in VN order, or E if absent    */
    const uint64_t *chan_dev;   /* [G][n][W]    1 = erased by the channel (LLRsChannel, BP_FULL.c:91)          */
} scldpc_batch_t;

/* Per-frame results, all int32 [G][64*W] on the device (lane = 64*w+b). */
typedef struct {
    int32_t *iters_dev;           /* iterations executed (full BP) / total over windows (window decoder)        */
    int32_t *residual_dev;        /* NumErasures returned by decodeBP / decodeBP_SW                             */
    int32_t *blocks_err_dev;      /* *num_blocks_err                                                           */
    int32_t *erasures_exp_dev;    /* *num_erasures_exp                                                         */
    int32_t *blocks_err_exp_dev;  /* *num_blocks_err_exp                                                       */
    int32_t *erasures_p1_dev;     /* *NumErasuresP1 (window decoder only; may be NULL)                         */
    uint64_t *erased_dev;         /* [G][n][W] VNerased after decoding (BP_FULL.c:94)                          */
    int32_t *rows_dev;            /* [G][max_rows][64*W][3] trajectory rows (deg1, dVNs, first_pos) or NULL     */
    int32_t max_rows;
} scldpc_bp_out_t;

const char *scldpc_last_error(void);
int scldpc_version(void);
/* "src=<hash> built=<date time> cuda=<version> arch=sm_100a"; <hash> = first 16 hex digits of sha256 over the .cu files of csrc (Makefile
 * order), common.cuh and this header -- the same value `make -C csrc print-hash` prints for the sources on disk */
const char *scldpc_build_info(void);
/* number of CUDA devices visible (0 => every compute call fails); never throws */
int scldpc_device_count(void);

/* ---- graph tables ------------------------------------------------------------------------------------ */
/* Builds vn_slot / cn_edge from vn_cn on the device, CN rows in the order generate_code appends them
 * (BP_FULL.c:1702-1716).  Replaces the CNdegree half of generate_code.  scratch_dev: int32 [G][nk]. */
int scldpc_graph_build_tables(const scldpc_dims_t *d, const scldpc_batch_t *b, int32_t *scratch_dev, void *stream);
/* Stream-ordered form without the host synchronisation of the call above: the validity flag (0 = fine, 1 = CN index out of
 * range, 2 = a CN with more than dc edges) is left in *err_dev (device int32) for the caller to read later.  Graphs drawn by
 * scldpc_graph_generate are valid by construction, so a Monte-Carlo loop that redraws its graphs every batch
 * (main_terminated, BP_FULL.c:2117-2143) never has to stop the device for them. */
int scldpc_graph_build_tables_async(const scldpc_dims_t *d, const scldpc_batch_t *b, int32_t *scratch_dev, int32_t *err_dev, void *stream);

/* On-device ensemble generation: the "Olmos random ensemble" of generate_code (BP_FULL.c:1656-1761) /
 * SC.gen_slots (SC.py:33-56): an independent uniform socket permutation per CN position.  Graph g of the batch
 * is realisation first_graph_id+g of stream `seed` (Philox4x32-10), independent of the batch / GPU layout.
 * The last argument selects the ensemble: 0 = semi-structured, 1 = its tail-biting variant SC.gen_slots_tail_biting
 * (SC.py:41-45, nk = L*cns_pos), 2 = protograph-based (sc_ldpc_protograph.py:6-20: per (position, portion, edge type) a
 * uniform permutation of the cns_pos CNs).  scratch_dev: sort keys, scldpc_graph_generate_scratch_bytes bytes. */
int scldpc_graph_generate(const scldpc_dims_t *d, int32_t *vn_cn_dev, uint64_t *scratch_dev, uint64_t seed,
                          uint64_t first_graph_id, int tail_biting, void *stream);
size_t scldpc_graph_generate_scratch_bytes(const scldpc_dims_t *d, int tail_biting);
/* Semi-structured ensemble for a PIECE of a longer chain: local position j of the piece is absolute position
 * first_position + j, and CN position p draws the same socket permutation whatever piece it is generated in -- the
 * streaming decoder (main_streaming / generate_code_pos, BP_FULL.c:1820-1856, :2003-2012) walks an unbounded chain in
 * overlapping pieces.  Scratch as for scldpc_graph_generate with ensemble 0. */
int scldpc_graph_generate_at(const scldpc_dims_t *d, int32_t *vn_cn_dev, uint64_t *scratch_dev, uint64_t seed,
                             uint64_t first_graph_id, uint32_t first_position, void *stream);

/* ---- channel ------------------------------------------------------------------------------------------ */
/* BEC realisations, bit-sliced (channel_doped, BP_FULL.c:1547-1574; PD.py:154, :174-192).  Lane f of graph g holds
 * frame first_frame_id+f (a multiple of 4) of Philox stream (seed, first_graph_id+g).  Hard doping: all VNs of positions doped_pos_host[] known.
 * Soft doping: the first soft_count_host[p] VNs of position soft_pos_host[p] known (int(alpha*M), PD.py:177). */
int scldpc_channel_generate(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                            int n_doped, const int32_t *soft_pos_host, const int32_t *soft_count_host, int n_soft,
                            uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id, void *stream);

/* Channel realisations for a piece of a longer chain (generate_channel_doped_circular, BP_FULL.c:1621-1654): local VN v is
 * VN first_vn_id + v of the stream, so overlapping pieces see the same erasures.  Hard doping only (local positions). */
int scldpc_channel_generate_at(const scldpc_dims_t *d, uint64_t *chan_dev, double eps, const int32_t *doped_pos_host,
                               int n_doped, uint64_t seed, uint64_t first_graph_id, uint32_t first_frame_id,
                               uint32_t first_vn_id, void *stream);

/* Packs byte-per-VN erasure patterns (host, [G][n_frames][n], 1 = erased) into chan_dev. */
int scldpc_channel_pack_host(const scldpc_dims_t *d, const uint8_t *erased_host, uint64_t *chan_dev, void *stream);

/* ---- decoders ----------------------------------------------------------------------------------------- */
size_t scldpc_bp_workspace_bytes(const scldpc_dims_t *d, uint32_t flags);

/* Full flooding BP over the BEC -- decodeBP (BP_FULL.c:900-1140, BP_TRAJ.c:901-1151).  max_it <= 0 means
 * unlimited (run until every frame has stalled or finished).  *iters_launched_host (optional) receives the number of
 * flooding iterations launched for the batch.
 * unscanned_head_cns > 0 -- simulate_sc_ldpc with is_bounded = False (PD.py:604-605,656): slots below
 * ignored_head_schedule*cns_per_pos are never scanned, they only decode when a removal leaves them with one user.  In BP
 * terms a CN below unscanned_head_cns that starts with exactly one erased neighbour keeps sending erasures.  0 = off. */
int scldpc_bp_full(const scldpc_dims_t *d, const scldpc_batch_t *b, int max_it, uint32_t flags,
                   int unscanned_head_cns, const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                   int *iters_launched_host, void *stream);

/* Per-position results of the last scldpc_bp_full / scldpc_bp_window call on this workspace, int32 [G][L][64*W] each:
 * erased VNs per position and accepted size-two stopping sets per position (get_deg_two_ss, BP_FULL.c:1227-1283: the
 * expurgated count of a position is pos_cnt - 2*pos_pairs).  These are what main_streaming / decodeBP_SW_circular
 * accumulate position by position (BP_FULL.c:1483-1497, :2015-2031). */
int scldpc_bp_position_counts(const scldpc_dims_t *d, uint32_t flags, void *workspace_dev, int32_t *pos_cnt_dev,
                              int32_t *pos_pairs_dev, void *stream);

/* Per-iteration moments of the trajectory rows of a scldpc_bp_full call with SCLDPC_F_TRAJECTORY, accumulated (+=) into
 * acc_dev int64 [max_rows][8]: per iteration t = (frames that executed t, frames with dVNs != 0, sum dVNs, sum dVNs^2,
 * sum deg_1_iter, sum deg_1_iter^2, sum first erased position, sum dVNs*deg_1_iter).  These are what the notebook derives
 * from bp_traj's text rows (BP_TRAJ.c:988,1051; NB cells 40-42: mean dVNs over non-zero entries, variance around the
 * mean-evolution curve with finished frames zero-padded) -- exact integers, additive over batches and ranks. */
int scldpc_bp_trajectory_moments(const scldpc_dims_t *d, const int32_t *rows_dev, const int32_t *iters_dev, int max_rows,
                                 int64_t *acc_dev, void *stream);

/* Stopping-set bookkeeping of simulate_sc_ldpc (PD.py:659-691) on the residual graph of a decode: per frame the "lost" VNs
 * (erased VNs of the positions with counted_pos_host[p] != 0; NULL = all) are split into the connected components
 * extract_stopping_sets would return (PD.py:1077-1095: two lost VNs are connected when they share a CN) and summarised as
 * out_dev int32 [G][64*W][4] = (num_lost, any component with more than 2 VNs, VNs in such components, VN positions such
 * components touch) -- num_lost, num_fuckups_truncated, num_lost_exp and len(lost_exp) of PD.py:671-689.
 * erased_dev: uint64 [G][n][W], e.g. scldpc_bp_out_t.erased_dev of the preceding scldpc_bp_full call. */
int scldpc_bp_stopping_sets(const scldpc_dims_t *d, const scldpc_batch_t *b, const uint64_t *erased_dev,
                            const uint8_t *counted_pos_host, int32_t *out_dev, void *stream);

/* Frame streams (lane recycling).  Each graph of the batch decodes frames 0 .. frames_per_graph-1 of its channel
 * stream (the same realisations scldpc_channel_generate produces for those frame ids) with unlimited-iteration full
 * BP; d->n_frames lanes per graph are used, and a lane whose frame has stopped is harvested and re-armed with the next
 * frame id, so stragglers do not hold the other lanes of their word idle.  Results are indexed by frame id,
 * int32 [G][frames_per_graph].  b->chan_dev is not used. */
typedef struct {
    int32_t frames_per_graph;        /* stream length per graph                                                */
    int32_t harvest_every;           /* iterations between harvests (<= 0: adapted to the iterations per frame) */
    uint32_t flags;                  /* SCLDPC_F_TERMINATED, SCLDPC_F_EXP_ALL, SCLDPC_F_MESSAGES               */
    int32_t n_doped, n_soft;
    const double *eps_host;          /* [G] erasure probability of each graph's channel                        */
    const int32_t *doped_pos_host, *soft_pos_host, *soft_count_host;   /* doping as in scldpc_channel_generate  */
    uint64_t seed, first_graph_id;
    int32_t max_it;                  /* iteration cap per frame, do {} while (iter < MaxNumIt) (BP_FULL.c:1066); <= 0: none.
                                        Needs the node-state sweeps (no SCLDPC_F_MESSAGES)                     */
} scldpc_stream_cfg_t;
typedef struct {
    int32_t *iters_dev, *residual_dev, *blocks_err_dev, *erasures_exp_dev, *blocks_err_exp_dev;
} scldpc_stream_out_t;
size_t scldpc_bp_stream_workspace_bytes(const scldpc_dims_t *d, uint32_t flags /* SCLDPC_F_MESSAGES or 0 */);
int scldpc_bp_stream(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg,
                     const scldpc_stream_out_t *out, void *workspace_dev, size_t workspace_bytes,
                     long long *iters_launched_host, void *stream);

/* Frame streams with checkpoints: one decode yields the results of every iteration cap of an ascending list.
 * On the BEC, flooding BP from the channel erasures is monotone and a stall is a fixed point, so the erased set a frame has
 * under cap T is the erased set of the unlimited decoder after min(T, stop) iterations.  A frame that reaches caps_host[k]
 * (k < n_caps-1) pauses until the next harvest, which records its statistics into slot k and lets it continue; when it
 * stops for good, its final statistics fill the slots it has not reached.  Slot k therefore equals a scldpc_bp_stream call
 * with cfg->max_it = caps_host[k], frame for frame (its iteration counts are min(iters_dev, caps_host[k])).
 * caps_host: 1 <= n_caps <= SCLDPC_MAX_CAPS strictly ascending values >= 1; only the last may be <= 0 (unlimited).
 * cfg->max_it must be 0 and SCLDPC_F_MESSAGES is not supported (node-state sweeps only).  The workspace comes from
 * scldpc_bp_stream_caps_workspace_bytes. */
#define SCLDPC_MAX_CAPS 16
typedef struct {
    int32_t *iters_dev;                 /* [G][B] iterations under the largest cap                               */
    int32_t *residual_dev, *blocks_err_dev, *erasures_exp_dev, *blocks_err_exp_dev;   /* [K][G][B] each      */
} scldpc_stream_caps_out_t;
size_t scldpc_bp_stream_caps_workspace_bytes(const scldpc_dims_t *d);
int scldpc_bp_stream_caps(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg,
                          const int32_t *caps_host, int n_caps, const scldpc_stream_caps_out_t *out,
                          void *workspace_dev, size_t workspace_bytes, long long *iters_launched_host, void *stream);

/* Frame streams with stopping-set records: simulate_sc_ldpc (PD.py:591-701) on unlimited BP with lane recycling.  Each frame
 * decodes to the peeling fixed point (the in-order sic_round scan, PD.py:656-657); its record is what
 * scldpc_bp_stopping_sets returns for it (PD.py:659-691): (num_lost, any component with more than 2 VNs, VNs in such
 * components, VN positions they touch), lost VNs being the erased VNs of the positions with counted_pos_host[p] != 0 (NULL =
 * all).  unscanned_head_cns > 0 is is_bounded = False (PD.py:604-606, :656) as in scldpc_bp_full: a CN below it that starts a
 * frame with exactly one erased neighbour never resolves it; it must not exceed the CNs the decoder sweeps
 * ((L+dv-1)*cns_pos with SCLDPC_F_TERMINATED, L*cns_pos without).  Frame f of graph g is the frame scldpc_bp_stream decodes,
 * and its iterations are what scldpc_bp_full(..., unscanned_head_cns) counts for it.  cfg->max_it must be 0 and
 * SCLDPC_F_MESSAGES is not supported (node-state sweeps only).  The workspace comes from
 * scldpc_bp_stream_stopping_sets_workspace_bytes. */
typedef struct {
    int32_t *iters_dev;     /* [G][B] iterations of each frame (unlimited BP)                                   */
    int32_t *records_dev;   /* [G][B][4] (num_lost, big component?, VNs in big components, positions they touch) */
} scldpc_stream_ss_out_t;
size_t scldpc_bp_stream_stopping_sets_workspace_bytes(const scldpc_dims_t *d);
int scldpc_bp_stream_stopping_sets(const scldpc_dims_t *d, const scldpc_batch_t *b, const scldpc_stream_cfg_t *cfg,
                                   const uint8_t *counted_pos_host /* [L], NULL = all */, int unscanned_head_cns,
                                   const scldpc_stream_ss_out_t *out, void *workspace_dev, size_t workspace_bytes,
                                   long long *iters_launched_host, void *stream);

/* scldpc_bp_stream with HOST buffers: graph tables vn_cn_host [G][n][dv] in, per-frame results int32
 * [G][frames_per_graph] out (any may be NULL); channel realisations are drawn on the device. */
int scldpc_stream_host(const scldpc_dims_t *d, const int32_t *vn_cn_host, const scldpc_stream_cfg_t *cfg,
                       int32_t *iters_host, int32_t *residual_host, int32_t *blocks_err_host, int32_t *erasures_exp_host,
                       int32_t *blocks_err_exp_host, long long *iters_launched_host);

/* Sliding-window BP -- decodeBP_SW (square: BP_SW.c:628-912; classical: BP_FULL.c:627-897).  init_it <= 0 means
 * max_it (BP_SW.c:2099-2102).  Without SCLDPC_F_TERMINATED the CN window is clipped at L*cns_pos (derived
 * non-terminated mode, SURVEY.md 8a-B2). */
int scldpc_bp_window(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                     const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                     int64_t *edge_updates_host, void *stream);

/* A range of windows of scldpc_bp_window, with the decoder state owned by the caller: windows [first_window, first_window +
 * n_windows) (n_windows < 0: to the end); pending_dev uint64 [G][n][W] is the second state plane of the node-state sweeps
 * (what every VN has been told so far; out->erased_dev holds what the CNs see).  resume == 0 initialises both planes from
 * the channel; resume != 0 continues from what the caller put there -- decodeBP_SW_circular (BP_FULL.c:1403-1500) decodes an
 * unbounded chain position by position, here piece by piece with the state of the overlap carried over.  Node-state sweeps
 * only.  Per-frame outputs and scldpc_bp_position_counts cover the whole piece; positions not yet decided are not final. */
int scldpc_bp_window_range(const scldpc_dims_t *d, const scldpc_batch_t *b, int W, int max_it, int init_it, uint32_t flags,
                           int first_window, int n_windows, uint64_t *pending_dev, int resume,
                           const scldpc_bp_out_t *out, void *workspace_dev, size_t workspace_bytes,
                           int64_t *edge_updates_host, void *stream);

/* Reference-facing convenience entry point with HOST buffers (what a maintainer would call in place of
 * generate_code + channel_doped + decodeBP, BP_FULL.c:2122-2133): uploads vn_cn_host [G][n][dv] and erased_host
 * [G][n_frames][n], decodes, and downloads the per-frame results (int32 [G][n_frames] each; any may be NULL) and
 * optionally the erased bitmaps (uint8 [G][n_frames][n]).  W == 0 selects full BP, W > 0 the window decoder.
 * All device memory is allocated and released inside the call. */
int scldpc_decode_host(const scldpc_dims_t *d, const int32_t *vn_cn_host, const uint8_t *erased_host, int W, int max_it,
                       int init_it, uint32_t flags, int32_t *iters_host, int32_t *residual_host,
                       int32_t *blocks_err_host, int32_t *erasures_exp_host, int32_t *blocks_err_exp_host,
                       int32_t *erasures_p1_host, uint8_t *vn_erased_host, int32_t *rows_host, int max_rows);

/* ---- peeling decoder with degree-one trajectory -------------------------------------------------------------- */
/* simulate_peeling_decoder_ldpc's per-frame loop (PD.py:740-785) for d->n_graphs graphs x d->n_frames frames:
 *   vn_cn_dev  [G][n][dv]  `transmissions` (SC.gen_slots, SC.py:53); CN indices run over n_cn_all CNs
 *   chan_dev   [G][n][W]   erased VNs, i.e. the Users that are generated (PD.py:154-163, :174-195 after doping)
 *   total_size             CNs the decoder sees: cns_per_pos * num_positions (PD.py:717-719); the rest are ignored
 *   num_steps              num_pd_steps = int(M * num_positions * (e + 0.1)) -- evaluate it in Python (PD.py:721)
 * Step s of global frame F = first_frame_id + g*n_frames + f picks the (u mod k)-th degree-one CN in ascending order,
 * u = scldpc_philox_picks(seed, F)[s], k = number of degree-one CNs (pick_random_deg_1_cn, PD.py:1022-1026).
 * Outputs: r1_dev int32 [G][n_frames][num_steps+1] (may be NULL), recovered_dev / n_erased_dev int32 [G][n_frames]
 * (plrs = (n_erased - recovered) / total_generated, PD.py:785). */
size_t scldpc_peel_workspace_bytes(const scldpc_dims_t *d, int n_cn_all, int total_size);
int scldpc_peel_trajectories(const scldpc_dims_t *d, const int32_t *vn_cn_dev, const uint64_t *chan_dev, int n_cn_all,
                             int total_size, int num_steps, uint64_t seed, uint64_t first_frame_id, int32_t *r1_dev,
                             int32_t *recovered_dev, int32_t *n_erased_dev, void *workspace_dev, size_t workspace_bytes,
                             void *stream);
/* calc_var_chunk (fl_scaling/est_scaling_params.py:131-138) fused on the device: for s < S, over the frames in order,
 * ssq[s] += (r1/M - theory[s]/M)^2 and counts[s] += 1 for frames with r1 != 0 (float64, same summation order as
 * np.nansum(axis=0)).  r1_dev has row_len columns. */
int scldpc_peel_variance_accumulate(const int32_t *r1_dev, int n_frames, int row_len, const double *theory_dev, int S,
                                    double M, double *ssq_dev, int64_t *counts_dev, void *stream);
/* The reduction behind DataFrame.corr() in calc_theta_explicit_ss_bounds / _ppd (fl_scaling/est_scaling_params.py:161-189,
 * :211-243): for the K sampled columns c_i = start + i*step of r1_dev [n_frames][row_len] (zeros are "missing"), accumulates
 * (+=) into acc_dev int64 [4][K][K] the pairwise-complete moments  N_ij = #{f: X_fi != 0 and X_fj != 0},
 * Sx_ij = sum_f X_fi [X_fj != 0], Sxx_ij = sum_f X_fi^2 [X_fj != 0], Sxy_ij = sum_f X_fi X_fj, from which
 * corr_ij = (N Sxy - Sx_ij Sx_ji) / sqrt((N Sxx_ij - Sx_ij^2)(N Sxx_ji - Sx_ji^2)).  Exact integers, additive over chunks and
 * ranks.  Works for peeling r1 trajectories and for the dVNs column of BP trajectory rows alike. */
int scldpc_pairwise_moments_accumulate(const int32_t *r1_dev, int n_frames, int row_len, int start, int step, int K,
                                       int64_t *acc_dev, void *stream);
/* the 32-bit draws behind the picks of one frame (host function; used to feed the reference the same pick sequence) */
void scldpc_philox_picks(uint64_t seed, uint64_t frame_id, int n, uint32_t *out_host);

/* ---- multi-GPU ------------------------------------------------------------------------------------------- */
/* Frames shard trivially (global graph / frame ids, no data-path collective); the one exchange is the sum of the final
 * counter or accumulator vectors -- what the reference does offline with awk / pickle sums over its per-process files
 * (NB:565, NB:1195, notebook cell 23).  nccl_comm: the caller's ncclComm_t; counters_dev: int64 [n_int64], reduced in
 * place on `stream`.  NCCL is resolved with dlopen at call time (no link-time dependency). */
int scldpc_allreduce_counters(void *nccl_comm, int64_t *counters_dev, int n_int64, void *stream);

/* ---- instrumentation ------------------------------------------------------------------------------------ */
/* The launch counter and the sampling state are per calling host thread (concurrent callers do not interfere).
 * kernels launched by the library (from this thread) since the last reset; scldpc_bp_sweep_stats: CN / VN positions swept by the last
 * scldpc_bp_full call on this workspace (wave tracking skips positions whose inputs did not change).  On the workspace
 * of a node-state scldpc_bp_stream call (flags SCLDPC_F_STREAM): out[0] = lane compactions done in the tails of the
 * graphs' streams, out[1] = frames they moved */
long long scldpc_launch_count(int reset);
/* Sampled CUDA-event timing of the two sweeps of every sample_every-th flooding iteration (on the launching
 * stream).  profile_end synchronises the device and returns per sample the iteration index and the CN / VN sweep
 * durations in milliseconds. */
int scldpc_bp_sweep_stats(const scldpc_dims_t *d, uint32_t flags, void *workspace_dev, long long *out_host);
int scldpc_profile_begin(int sample_every, int max_samples);
int scldpc_profile_end(int *n_samples, int *iter_idx, float *cn_ms, float *vn_ms, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* SCLDPC_H */
