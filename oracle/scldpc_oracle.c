/*
 * scldpc_oracle.c -- CPU restatement of the reference BEC decoders for SC-LDPC codes.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the *checker* for the CUDA path: it may be compiled, linked
 * and called by tests/, __graft_entry__.smoke() and the cpu_baseline / --impl reference legs of bench.py
 * and by nothing else.  The product library (libscldpc.so) never links or calls it.
 *
 * Parity status: PINNED.  Every function below is checked (tests/test_oracle_golden.py) against the
 * unmodified reference C code compiled from /root/reference by oracle/build_ref.py (same glibc random()
 * stream => identical graphs, channels, decisions, counters and trajectory rows), and against the golden
 * vectors under tests/golden/ that were generated from that compiled reference.
 *
 * Each function cites the reference lines it follows.  Abbreviations (SURVEY.md):
 *   BP_FULL.c = simulators_sc_ldpc/bp_decoding/SC_LDPC_Simulator_BPDecoder_BEC_full_BP_LimIter_OlmosRandomEnsemble.c
 *   BP_SW.c   = simulators_sc_ldpc/bp_decoding/SC_LDPC_Simulator_BPDecoder_BEC_SlidingWindow_LimIter_OlmosRandomEnsemble.c
 *   BP_TRAJ.c = simulators_sc_ldpc/bp_decoding/trajectories_SC_LDPC_Simulator_BPDecoder_BEC_full_BP_OlmosRandomEnsemble.c
 *   PD.py     = simulators_sc_ldpc/peeling_decoding/peeling_decoding.py
 *
 * Differences from the reference are representational only: sizes are run-time arguments instead of
 * #defines, adjacency lives in caller-provided flat arrays instead of file-scope tables, and the reverse
 * edge of a message is looked up in a precomputed table instead of the reference's linear search
 * (BP_FULL.c:956, :997, :1017) -- the graphs have no parallel edges, so both find the same edge.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------------- */
/* Graph tables                                                                                       */
/* ------------------------------------------------------------------------------------------------- */

/* CN adjacency in the order generate_code appends it (BP_FULL.c:1702-1716): VNs ascending, edges ascending.
 * vn_cn[n][dv] -> cn_deg[nk], cn_vn[nk][dc] (neighbour VN), cn_ei[nk][dc] (edge index at that VN),
 * vn_slot[n][dv] (slot of edge (v,i) in its CN row).  Returns 0, or -1 if a CN would exceed degree dc. */
int orc_build_cn(int n, int nk, int dv, int dc, const int *vn_cn, int *cn_deg, int *cn_vn, int *cn_ei, int *vn_slot)
{
    memset(cn_deg, 0, sizeof(int) * (size_t)nk);
    for (int v = 0; v < n; v++)
        for (int i = 0; i < dv; i++) {
            int c = vn_cn[(size_t)v * dv + i];
            if (c < 0 || c >= nk || cn_deg[c] >= dc) return -1;
            int j = cn_deg[c]++;
            cn_vn[(size_t)c * dc + j] = v;
            cn_ei[(size_t)c * dc + j] = i;
            vn_slot[(size_t)v * dv + i] = j;
        }
    return 0;
}

/* generate_code (BP_FULL.c:1656-1761): for each of the L+dv-1 CN positions an in-place Fisher-Yates pass over
 * perm_code (state carried over between positions, frames; reset to the identity per epsilon point by
 * inizio_sim, BP_FULL.c:308-311) with ipick = i + random() % (len - i) (:1684); socket -> CN is perm/dc (:1693);
 * VN t of position p takes socket dv*t+i of CN position p+i (:1712).  Uses glibc random() like the reference
 * (unif_int, BP_FULL.c:373-381), so the same srandom() seed gives the same graph. */
void orc_generate_code(int L, int vns_pos, int cns_pos, int dv, int dc, int *perm_code, int *vn_cn)
{
    int len = cns_pos * dc;
    int npos = L + dv - 1;
    int *inter = (int *)malloc(sizeof(int) * (size_t)npos * len);
    for (int pos = 0; pos < npos; pos++) {
        for (int i = 0; i < len; i++) {
            int ipick = i + (int)(random() % (len - i));
            int t = perm_code[i];
            perm_code[i] = perm_code[ipick];
            perm_code[ipick] = t;
        }
        for (int i = 0; i < len; i++)
            inter[(size_t)pos * len + i] = pos * cns_pos + (int)((double)perm_code[i] / dc);
    }
    for (int pos = 0; pos < L; pos++)
        for (int t = 0; t < vns_pos; t++) {
            int v = pos * vns_pos + t;
            for (int i = 0; i < dv; i++)
                vn_cn[(size_t)v * dv + i] = inter[(size_t)(pos + i) * len + dv * t + i];
        }
    free(inter);
}

/* channel_doped (BP_FULL.c:1547-1574) with unif_ch = random()/RAND_MAX (:360-371): erased iff u < eps;
 * every VN of a doped position is forced known. */
void orc_channel_doped(int n, double eps, int vns_pos, int num_doped, const int *doped, int *chan)
{
    for (int j = 0; j < n; j++) {
        double u = (double)random() / RAND_MAX;
        chan[j] = (u >= eps) ? 0 : 1;
    }
    for (int d = 0; d < num_doped; d++)
        for (int j = doped[d] * vns_pos; j < (doped[d] + 1) * vns_pos; j++) chan[j] = 0;
}

/* is_position_doped_streaming (BP_FULL.c:1589-1612): periodic doping, period = last doped position + 1. */
int orc_is_position_doped_streaming(int pos, int num_doped, const int *doped)
{
    if (num_doped == 0) return 0;
    int period = doped[num_doped - 1] + 1;
    int r = pos % period;
    for (int d = 0; d < num_doped; d++)
        if (doped[d] == r) return 1;
    return 0;
}

/* ------------------------------------------------------------------------------------------------- */
/* Shared pieces of the decoders                                                                      */
/* ------------------------------------------------------------------------------------------------- */

typedef struct {
    int n, nk, dv, dc;
    const int *vn_cn, *cn_deg, *cn_vn, *cn_ei, *vn_slot, *chan;
    int *Lji; /* [n][dv]   VN j -> CN along edge i      */
    int *Lij; /* [nk][dc]  CN i -> VN along slot j      */
} orc_state;

/* CN update for CNs [c0,c1) (BP_FULL.c:943-968 / BP_SW.c:711-730).  If resolved != NULL also runs the
 * degree-one counter with its latch (BP_FULL.c:935-979) and returns deg_1_iter. */
static int cn_sweep(orc_state *s, int c0, int c1, char *resolved)
{
    int dv = s->dv, dc = s->dc, deg1 = 0;
    for (int c = c0; c < c1; c++) {
        int deg = s->cn_deg[c], num_out_resolved = 0;
        for (int j = 0; j < deg; j++) {
            int erasure = 0;
            for (int l = 0; l < deg; l++)
                if (l != j) erasure += s->Lji[(size_t)s->cn_vn[(size_t)c * dc + l] * dv + s->cn_ei[(size_t)c * dc + l]];
            if (erasure > 0) s->Lij[(size_t)c * dc + j] = 1;
            else { s->Lij[(size_t)c * dc + j] = 0; num_out_resolved++; }
        }
        if (resolved && !resolved[c] && num_out_resolved > 0) {
            if (num_out_resolved == 1) deg1++;
            resolved[c] = 1;
        }
    }
    return deg1;
}

/* VN update for VNs [v0,v1) (BP_FULL.c:985-1005 / BP_SW.c:735-755). */
static void vn_sweep(orc_state *s, int v0, int v1)
{
    int dv = s->dv, dc = s->dc;
    for (int v = v0; v < v1; v++)
        for (int i = 0; i < dv; i++) {
            int erasure = 0;
            for (int l = 0; l < dv; l++)
                if (l != i) erasure += s->Lij[(size_t)s->vn_cn[(size_t)v * dv + l] * dc + s->vn_slot[(size_t)v * dv + l]];
            s->Lji[(size_t)v * dv + i] = (erasure < dv - 1 || s->chan[v] == 0) ? 0 : 1;
        }
}

/* a-posteriori erasure of VN v (BP_FULL.c:1011-1024). */
static int vn_erased(const orc_state *s, int v)
{
    int dv = s->dv, dc = s->dc, erasure = 0;
    for (int i = 0; i < dv; i++)
        erasure += s->Lij[(size_t)s->vn_cn[(size_t)v * dv + i] * dc + s->vn_slot[(size_t)v * dv + i]];
    erasure += s->chan[v];
    return erasure == dv + 1;
}

/* Size-two stopping-set expurgation for one position (BP_FULL.c:1075-1125; identical text at BP_SW.c:857-902).
 * Returns the expurgated erasure count of the position; *num_pos gets the plain count. */
static int expurgate_pos(const orc_state *s, const unsigned char *erased, int vnpos, int vns_pos, int *num_pos)
{
    int dv = s->dv, dc = s->dc, exp_pos = 0, plain = 0;
    for (int a = 0; a < vns_pos; a++) {
        int vn_a = vnpos * vns_pos + a;
        if (!erased[vn_a]) continue;
        exp_pos++; plain++;
        for (int b = a + 1; b < vns_pos; b++) {
            int vn_b = vnpos * vns_pos + b;
            if (!erased[vn_b]) continue;
            int same_connections = 1, others_recovered = 1;
            for (int ac = 0; ac < dv; ac++) {
                int aux_a = s->vn_cn[(size_t)vn_a * dv + ac], conn_to_vn_b = 0;
                for (int cc = 0; cc < s->cn_deg[aux_a]; cc++) {
                    int cur = s->cn_vn[(size_t)aux_a * dc + cc];
                    if (cur == vn_b) conn_to_vn_b = 1;
                    else if (cur != vn_a && erased[cur]) others_recovered = 0;
                }
                if (!conn_to_vn_b) { same_connections = 0; break; }
                if (!others_recovered) break;
            }
            if (same_connections && others_recovered) exp_pos -= 2;
        }
    }
    *num_pos = plain;
    return exp_pos;
}

/* Per-position erasure counts and expurgated counts (get_deg_two_ss, BP_FULL.c:1227-1283) of a decided frame:
 * plain[p] = erased VNs of position p, exp[p] = plain[p] - 2 * (accepted size-two stopping sets of position p). */
void orc_position_counts(int n, int nk, int L, int vns_pos, int dv, int dc, const int *vn_cn, const int *cn_deg,
                         const int *cn_vn, const unsigned char *erased, int *plain, int *exp_cnt)
{
    orc_state s = { n, nk, dv, dc, vn_cn, cn_deg, cn_vn, NULL, NULL, NULL, NULL, NULL };
    for (int p = 0; p < L; p++) exp_cnt[p] = expurgate_pos(&s, erased, p, vns_pos, &plain[p]);
}

/* ------------------------------------------------------------------------------------------------- */
/* decodeBP: full flooding BP (BP_FULL.c:900-1140, BP_TRAJ.c:901-1151)                                */
/* ------------------------------------------------------------------------------------------------- */
/* rows (optional): int[max_rows][3] = (deg_1_iter, NumErasuresPrec-NumErasures, first_erased/VNsPos), one row per
 * executed iteration (BP_TRAJ.c:988,:1051).  *iters = number of executed iterations.
 * Lji_out/Lij_edge_out (optional): final messages, both indexed by VN edge [n][dv].
 * Returns NumErasures. */
int orc_decode_bp(int n, int nk, int L, int vns_pos, int cns_pos, int dv, int dc,
                  const int *vn_cn, const int *cn_deg, const int *cn_vn, const int *cn_ei, const int *vn_slot,
                  const int *chan, int max_it, int is_term,
                  unsigned char *erased, int *iters, int *blocks_err, int *erasures_exp, int *blocks_err_exp,
                  int *rows, int max_rows, int *Lji_out, int *Lij_edge_out)
{
    orc_state s = { n, nk, dv, dc, vn_cn, cn_deg, cn_vn, cn_ei, vn_slot, chan, NULL, NULL };
    s.Lji = (int *)malloc(sizeof(int) * (size_t)n * dv);
    s.Lij = (int *)calloc((size_t)nk * dc, sizeof(int));
    char *resolved = (char *)calloc((size_t)nk, 1);
    int NumErasures = 0, NumErasuresPrec = n, iter = 0, executed = 0;

    for (int v = 0; v < n; v++)                               /* BP_FULL.c:913-917 */
        for (int i = 0; i < dv; i++) s.Lji[(size_t)v * dv + i] = chan[v];
    int cn_lim = is_term ? nk : L * cns_pos;                  /* BP_TRAJ.c:944-948 */
    if (!is_term)                                             /* BP_TRAJ.c:922-925 */
        for (int c = L * cns_pos; c < nk; c++)
            for (int j = 0; j < cn_deg[c]; j++) s.Lij[(size_t)c * dc + j] = 1;

    do {
        int deg1 = cn_sweep(&s, 0, cn_lim, resolved);
        vn_sweep(&s, 0, n);
        int first_erased = n;
        NumErasures = 0;
        for (int v = 0; v < n; v++) {                          /* BP_TRAJ.c:1017-1045 */
            if (vn_erased(&s, v)) { erased[v] = 1; NumErasures++; if (v < first_erased) first_erased = v; }
            else erased[v] = 0;
        }
        if (rows && executed < max_rows) {
            rows[executed * 3 + 0] = deg1;
            rows[executed * 3 + 1] = NumErasuresPrec - NumErasures;
            rows[executed * 3 + 2] = first_erased / vns_pos;
        }
        executed++;
        if (NumErasures == 0) break;                           /* BP_FULL.c:1044-1045 */
        if (NumErasures == NumErasuresPrec) break;
        NumErasuresPrec = NumErasures;
        iter++;
    } while (iter < max_it);                                   /* BP_FULL.c:1065 */

    /* Expurgation: blocks in error = positions with any erased VN; the expurgated statistics take only the
     * FIRST position with a positive expurgated count (is_first_printed, BP_FULL.c:1074,1126-1131). */
    *blocks_err = 0; *erasures_exp = 0; *blocks_err_exp = 0;
    int first_printed = 0;
    for (int p = 0; p < L; p++) {
        int plain, e = expurgate_pos(&s, erased, p, vns_pos, &plain);
        if (plain > 0) *blocks_err += 1;
        if (e > 0 && !first_printed) { first_printed = 1; *erasures_exp += e; *blocks_err_exp += 1; }
    }
    if (iters) *iters = executed;
    if (Lji_out) memcpy(Lji_out, s.Lji, sizeof(int) * (size_t)n * dv);
    if (Lij_edge_out)
        for (int v = 0; v < n; v++)
            for (int i = 0; i < dv; i++)
                Lij_edge_out[(size_t)v * dv + i] = s.Lij[(size_t)vn_cn[(size_t)v * dv + i] * dc + vn_slot[(size_t)v * dv + i]];
    free(s.Lji); free(s.Lij); free(resolved);
    return NumErasures;
}

/* ------------------------------------------------------------------------------------------------- */
/* decodeBP_SW: sliding-window BP (square window BP_SW.c:628-912, classical window BP_FULL.c:627-897)  */
/* ------------------------------------------------------------------------------------------------- */
/* square=1: VN window [posW, posW+W), L windows, first window capped by init_it (BP_SW.c:672-703).
 * square=0: VN window [max(posW-ms,0), posW+W) (W+posW positions while posW<=ms), L+ms windows, decisions only
 *           when posW>=ms, every window capped by max_it (BP_FULL.c:668-690,:745).
 * is_term=0 is the DERIVED non-terminated mode (SURVEY.md section 8a row B2 / App. A-17, by analogy with
 * BP_TRAJ.c:922-925,944-948): the CN window is clipped at L*cns_pos and the excluded CNs keep Lij = 1.
 * win_iters (optional) int[number of windows]: iterations executed in each window.
 * Returns NumErasures (sum over windows of the decided position's erasures, BP_SW.c:841). */
int orc_decode_bp_sw(int n, int nk, int L, int W, int vns_pos, int cns_pos, int dv, int dc,
                     const int *vn_cn, const int *cn_deg, const int *cn_vn, const int *cn_ei, const int *vn_slot,
                     const int *chan, int max_it, int init_it, int square, int is_term,
                     unsigned char *erased, int *erasures_p1, int *blocks_err, int *erasures_exp, int *blocks_err_exp,
                     int *win_iters, int *Lji_out, int *Lij_edge_out)
{
    orc_state s = { n, nk, dv, dc, vn_cn, cn_deg, cn_vn, cn_ei, vn_slot, chan, NULL, NULL };
    s.Lji = (int *)malloc(sizeof(int) * (size_t)n * dv);
    s.Lij = (int *)malloc(sizeof(int) * (size_t)nk * dc);
    int ms = dv - 1, NumErasures = 0;
    int cn_clip = is_term ? nk : L * cns_pos;

    for (int v = 0; v < n; v++)                               /* BP_SW.c:650-654 */
        for (int i = 0; i < dv; i++) s.Lji[(size_t)v * dv + i] = chan[v];
    for (size_t k = 0; k < (size_t)nk * dc; k++) s.Lij[k] = 1; /* BP_SW.c:655-659 */
    memset(erased, 0, (size_t)n);                             /* generate_code zeroes VNerased, BP_FULL.c:1707 */

    *erasures_p1 = 0; *blocks_err = 0; *erasures_exp = 0; *blocks_err_exp = 0;
    int nwin = square ? L : L + ms;
    for (int posW = 0; posW < nwin; posW++) {
        int StartCN = posW * cns_pos, EndCN = StartCN + W * cns_pos, StartVN, EndVN;
        if (EndCN > cn_clip) EndCN = cn_clip;
        if (square) { StartVN = posW * vns_pos; EndVN = StartVN + W * vns_pos; }
        else if (posW <= ms) { StartVN = 0; EndVN = (W + posW) * vns_pos; }
        else { StartVN = (posW - ms) * vns_pos; EndVN = StartVN + (W + ms) * vns_pos; }
        if (EndVN > n) EndVN = n;
        int iter = 0, executed = 0, NumErasuresPos = 0, NumErasuresTerm, NumErasuresPrecTerm = n;
        int NumIt = (square && posW == 0) ? init_it : max_it;  /* BP_SW.c:699-702 */
        do {
            NumErasuresPos = 0; NumErasuresTerm = 0;
            cn_sweep(&s, StartCN, EndCN, NULL);
            vn_sweep(&s, StartVN, EndVN);
            if (square || posW >= ms)                          /* BP_FULL.c:745 */
                for (int v = StartVN; v < StartVN + vns_pos; v++) {
                    if (vn_erased(&s, v)) { erased[v] = 1; NumErasuresPos++; } else erased[v] = 0;
                }
            for (int v = StartVN; v < EndVN; v++) NumErasuresTerm += vn_erased(&s, v);   /* BP_SW.c:791-809 */
            executed++;
            if (NumErasuresTerm == 0) break;                   /* BP_SW.c:815-816 */
            if (NumErasuresTerm == NumErasuresPrecTerm) break;
            NumErasuresPrecTerm = NumErasuresTerm;
            iter++;
        } while (iter < NumIt);
        if (win_iters) win_iters[posW] = executed;
        NumErasures += NumErasuresPos;                          /* BP_SW.c:841-847 */
        if (NumErasuresPos > 0) *blocks_err += 1;
        if (posW >= ms && posW <= W - 2) *erasures_p1 += NumErasuresPos;
    }
    for (int p = 0; p < L; p++) {                               /* BP_SW.c:857-908: ALL positions are added */
        int plain, e = expurgate_pos(&s, erased, p, vns_pos, &plain);
        if (e > 0) { *erasures_exp += e; *blocks_err_exp += 1; }
    }
    if (Lji_out) memcpy(Lji_out, s.Lji, sizeof(int) * (size_t)n * dv);
    if (Lij_edge_out)
        for (int v = 0; v < n; v++)
            for (int i = 0; i < dv; i++)
                Lij_edge_out[(size_t)v * dv + i] = s.Lij[(size_t)vn_cn[(size_t)v * dv + i] * dc + vn_slot[(size_t)v * dv + i]];
    free(s.Lji); free(s.Lij);
    return NumErasures;
}

/* ------------------------------------------------------------------------------------------------- */
/* Peeling decoder with degree-one trajectory (PD.py:705-789, pick_random_deg_1_cn PD.py:1022-1026)    */
/* ------------------------------------------------------------------------------------------------- */
/* vn_cn[n_vn][l]  : `transmissions` (CN index per edge; indices >= total_size are the ignored tail CNs)
 * erased[n_vn]    : VNs that generate a User (PD.py:154-163 / :174-195 after doping)
 * picks[num_steps]: 32-bit uniform draws; step s with k degree-one CNs picks the (picks[s] % k)-th smallest CN
 *                   index -- the injected replacement of random.choice(np.flatnonzero(r == 1)) (PD.py:1023-1026).
 * r1[num_steps+1] : number of degree-one CNs after each step (PD.py:758,:767,:781).
 * Returns the number of recovered (peeled) VNs. */
int orc_peel_trajectory(int n_vn, int l, int total_size, int n_cn_all, const int *vn_cn, const unsigned char *erased,
                        int num_steps, const uint32_t *picks, int64_t *r1)
{
    int *r = (int *)calloc((size_t)n_cn_all, sizeof(int));
    /* residual graph restricted to erased VNs: XOR of neighbour ids identifies the last remaining VN of a CN */
    uint32_t *xr = (uint32_t *)calloc((size_t)n_cn_all, sizeof(uint32_t));
    unsigned char *alive = (unsigned char *)malloc((size_t)n_vn);
    memcpy(alive, erased, (size_t)n_vn);
    for (int v = 0; v < n_vn; v++)
        if (erased[v])
            for (int i = 0; i < l; i++) { int c = vn_cn[(size_t)v * l + i]; r[c]++; xr[c] ^= (uint32_t)v; }
    int recovered = 0;
    int64_t cnt1 = 0;
    for (int t = 0; t < total_size; t++) cnt1 += (r[t] == 1);   /* PD.py:756-758 */
    r1[0] = cnt1;
    for (int step = 0; step < num_steps; step++) {
        if (cnt1 == 0) { r1[step + 1] = r1[step]; continue; }   /* PD.py:765-767 */
        int64_t k = picks[step] % (uint64_t)cnt1;
        int m = -1;
        for (int t = 0; t < total_size; t++)
            if (r[t] == 1 && k-- == 0) { m = t; break; }
        int v = (int)xr[m];                                     /* head(schedule[m]) -- the only user left, PD.py:769 */
        alive[v] = 0; recovered++;
        for (int i = 0; i < l; i++) {                           /* PD.py:771-780 */
            int c = vn_cn[(size_t)v * l + i];
            xr[c] ^= (uint32_t)v;
            if (c < total_size) { if (r[c] == 1) cnt1--; r[c]--; if (r[c] == 1) cnt1++; }
            else r[c]--;
        }
        r1[step + 1] = cnt1;                                    /* PD.py:781 */
    }
    free(r); free(xr); free(alive);
    return recovered;
}

/* orc_peel_trajectory with the same inputs and outputs, O(log total_size) per step instead of O(total_size): the
 * degree-one indicator of the CNs [0, total_size) is kept in a Fenwick tree (1-based, fw[i] = number of degree-one CNs
 * in (i - lowbit(i), i]), and "the k-th degree-one CN in ascending order" is the usual top-down descent over it.
 * Written from the PD.py semantics above, not from the kernel's bitmap hierarchy, so that it stays an independent check;
 * tests/test_peel_oracle_cpu.py holds it to orc_peel_trajectory. */
static void fw_add(int *fw, int n, int t, int d)
{
    for (int i = t + 1; i <= n; i += i & -i) fw[i] += d;
}

static int fw_select(const int *fw, int n, int64_t k)   /* 0-based index of the (k+1)-th set position */
{
    int pos = 0, top = 1;
    while (top * 2 <= n) top *= 2;
    for (int b = top; b; b >>= 1)
        if (pos + b <= n && fw[pos + b] <= k) { pos += b; k -= fw[pos]; }
    return pos;
}

int orc_peel_trajectory_fast(int n_vn, int l, int total_size, int n_cn_all, const int *vn_cn, const unsigned char *erased,
                             int num_steps, const uint32_t *picks, int64_t *r1)
{
    int *r = (int *)calloc((size_t)n_cn_all, sizeof(int));
    uint32_t *xr = (uint32_t *)calloc((size_t)n_cn_all, sizeof(uint32_t));
    int *fw = (int *)calloc((size_t)total_size + 1, sizeof(int));
    for (int v = 0; v < n_vn; v++)
        if (erased[v])
            for (int i = 0; i < l; i++) { int c = vn_cn[(size_t)v * l + i]; r[c]++; xr[c] ^= (uint32_t)v; }
    int64_t cnt1 = 0;
    for (int t = 0; t < total_size; t++)                         /* linear-time build: push each node into its parent */
        if (r[t] == 1) { fw[t + 1] += 1; cnt1++; }
    for (int i = 1; i <= total_size; i++) {
        int p = i + (i & -i);
        if (p <= total_size) fw[p] += fw[i];
    }
    r1[0] = cnt1;
    int recovered = 0;
    for (int step = 0; step < num_steps; step++) {
        if (cnt1 == 0) { r1[step + 1] = r1[step]; continue; }
        int m = fw_select(fw, total_size, (int64_t)(picks[step] % (uint64_t)cnt1));
        int v = (int)xr[m];
        recovered++;
        for (int i = 0; i < l; i++) {
            int c = vn_cn[(size_t)v * l + i];
            xr[c] ^= (uint32_t)v;
            r[c]--;
            if (c < total_size) {
                if (r[c] == 1) { fw_add(fw, total_size, c, 1); cnt1++; }
                else if (r[c] == 0) { fw_add(fw, total_size, c, -1); cnt1--; }
            }
        }
        r1[step + 1] = cnt1;
    }
    free(r); free(xr); free(fw);
    return recovered;
}

/* Peeling to the fixed point = residual of unlimited flooding BP (simulate_sc_ldpc's sic_round scan,
 * PD.py:270-320,:656-657, reaches the same maximal stopping set; SURVEY.md section 3.5).  Slots are scanned from
 * scan_lo = ignored_head_schedule*cns_per_pos up to cn_hi = total_size (PD.py:656); a cascade
 * (subtract_interference, PD.py:294-320) may also decode a slot below scan_lo when a removal leaves it with one
 * user (the only bound there is slot_idx <= t), but never a slot >= cn_hi.  lost[v] = 1 for erased VNs never
 * resolved. */
void orc_peel_fixed_point(int n_vn, int l, int n_cn_all, int scan_lo, int cn_hi, const int *vn_cn,
                          const unsigned char *erased, unsigned char *lost)
{
    int *r = (int *)calloc((size_t)n_cn_all, sizeof(int));
    uint32_t *xr = (uint32_t *)calloc((size_t)n_cn_all, sizeof(uint32_t));
    int *stack = (int *)malloc(sizeof(int) * ((size_t)n_cn_all + (size_t)n_vn * l + 1));
    int sp = 0;
    memcpy(lost, erased, (size_t)n_vn);
    for (int v = 0; v < n_vn; v++)
        if (erased[v])
            for (int i = 0; i < l; i++) { int c = vn_cn[(size_t)v * l + i]; r[c]++; xr[c] ^= (uint32_t)v; }
    for (int c = scan_lo; c < cn_hi; c++) if (r[c] == 1) stack[sp++] = c;
    while (sp) {
        int c = stack[--sp];
        if (r[c] != 1) continue;
        int v = (int)xr[c];
        lost[v] = 0;
        for (int i = 0; i < l; i++) {
            int c2 = vn_cn[(size_t)v * l + i];
            r[c2]--; xr[c2] ^= (uint32_t)v;
            if (r[c2] == 1 && c2 < cn_hi) stack[sp++] = c2;
        }
    }
    free(r); free(xr); free(stack);
}
