/* CPU oracle for kernel (a): edge_index -> canonical CSR.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/sage_oracle.py header).  Plain C restatement of
 * the CSR oracle in SURVEY.md 8(c): order = lexsort((src, dst)) (stable), col = src[order],
 * rowptr = exclusive cumsum(bincount(dst)), perm = order, inv_deg = 1/max(deg,1).
 * It is what PyG's SAGEConv effectively consumes after sort_edge_index(sort_by_row=False);
 * the reference's call site is src/deep_fem_uav_wing/gnn/model.py:90 (edge_index int64 [2,E]
 * produced at gnn/dataset.py:63).
 *
 * Two stable counting sorts (LSD): first by src, then by dst.  O(E + N), no comparison sort.
 * Also hosts a plain-C aggregation that mirrors the arithmetic of the gather kernel, for the oracle and kernel tests.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* returns 0 ok, 1 bad index, 2 alloc failure */
int oracle_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int by_src,
                     int32_t* rowptr, int32_t* col, int32_t* perm, float* inv_deg) {
    const int64_t* src = edge_index;
    const int64_t* dst = edge_index + E;
    if (by_src) { const int64_t* t = src; src = dst; dst = t; }
    for (int64_t e = 0; e < E; ++e)
        if (src[e] < 0 || src[e] >= N || dst[e] < 0 || dst[e] >= N) return 1;

    int64_t* cnt = (int64_t*)calloc((size_t)N + 1, sizeof(int64_t));
    int32_t* tmp = (int32_t*)malloc(sizeof(int32_t) * (size_t)(E > 0 ? E : 1));
    if (!cnt || !tmp) { free(cnt); free(tmp); return 2; }

    /* pass 1: stable counting sort of edge ids by src */
    for (int64_t e = 0; e < E; ++e) cnt[src[e] + 1]++;
    for (int64_t i = 0; i < N; ++i) cnt[i + 1] += cnt[i];
    for (int64_t e = 0; e < E; ++e) tmp[cnt[src[e]]++] = (int32_t)e;

    /* pass 2: stable counting sort of that sequence by dst */
    memset(cnt, 0, sizeof(int64_t) * ((size_t)N + 1));
    for (int64_t e = 0; e < E; ++e) cnt[dst[e] + 1]++;
    for (int64_t i = 0; i < N; ++i) cnt[i + 1] += cnt[i];
    for (int64_t i = 0; i <= N; ++i) rowptr[i] = (int32_t)cnt[i];
    for (int64_t i = 0; i < N; ++i) {
        int64_t d = cnt[i + 1] - cnt[i];
        inv_deg[i] = 1.0f / (float)(d > 0 ? d : 1);
    }
    for (int64_t k = 0; k < E; ++k) {
        int32_t e = tmp[k];
        int64_t p = cnt[dst[e]]++;
        perm[p] = e;
        col[p] = (int32_t)src[e];
    }
    free(cnt);
    free(tmp);
    return 0;
}

/* Mean / sum aggregation with every form of the device kernel (dfw_aggregate.cu), step by step in its arithmetic:
 *   acc = 0;  per edge k of row i, in CSR order:  acc = fmaf(x[col[k]], src_scale[col[k]], acc)   (src_scale given)
 *                                                 acc = acc + x[col[k]]                             (otherwise)
 *   out[i] = fmaf(acc, sc_i, addend[i])  with an addend,  acc * sc_i  without;  sc_i = row_scale[i], or 1 when NULL.
 * All in fp32 with round-to-nearest-even; fmaf is libm's correctly rounded fused multiply-add, and the Makefile builds with
 * -ffp-contract=off so that no other multiply and add are fused.  A bf16 tensor is passed as its exact fp32 widening and
 * the bf16 result is rounded by the caller.  x has as many rows as col indexes (more than N_rows for a rectangular CSR).
 * Rows are independent, so contiguous row ranges run on several host threads (pthreads; no OpenMP runtime in the
 * image): every row is still summed sequentially in CSR order by one thread, so the result does not depend on the
 * thread count. */
#include <math.h>
#include <pthread.h>
#include <unistd.h>

typedef struct {
    const int32_t* rowptr; const int32_t* col; const float* row_scale; const float* src_scale; const float* x;
    const float* addend; float* out;
    int64_t r0, r1, H;
} agg_job;

static void* agg_rows(void* arg) {
    const agg_job* j = (const agg_job*)arg;
    const int64_t H = j->H;
    for (int64_t i = j->r0; i < j->r1; ++i) {
        float* o = j->out + i * H;
        for (int64_t h = 0; h < H; ++h) o[h] = 0.0f;
        for (int32_t k = j->rowptr[i]; k < j->rowptr[i + 1]; ++k) {
            const float* r = j->x + (int64_t)j->col[k] * H;
            if (j->src_scale) {
                const float s = j->src_scale[j->col[k]];
                for (int64_t h = 0; h < H; ++h) o[h] = fmaf(r[h], s, o[h]);
            } else {
                for (int64_t h = 0; h < H; ++h) o[h] += r[h];
            }
        }
        const float sc = j->row_scale ? j->row_scale[i] : 1.0f;
        if (j->addend) {
            const float* a = j->addend + i * H;
            for (int64_t h = 0; h < H; ++h) o[h] = fmaf(o[h], sc, a[h]);
        } else {
            for (int64_t h = 0; h < H; ++h) o[h] *= sc;
        }
    }
    return 0;
}

void oracle_csr_aggregate_ex_f32(const int32_t* rowptr, const int32_t* col, const float* row_scale, const float* src_scale,
                                 const float* x, const float* addend, float* out, int64_t N_rows, int64_t H) {
    long nproc = sysconf(_SC_NPROCESSORS_ONLN);
    int T = (int)(nproc < 1 ? 1 : (nproc > 32 ? 32 : nproc));
    if (N_rows * H < (1 << 22)) T = 1;
    agg_job jobs[32];
    pthread_t th[32];
    const int64_t per = (N_rows + T - 1) / T;
    for (int t = 0; t < T; ++t) {
        agg_job j = {rowptr, col, row_scale, src_scale, x, addend, out,
                     t * per < N_rows ? t * per : N_rows, (t + 1) * per < N_rows ? (t + 1) * per : N_rows, H};
        jobs[t] = j;
    }
    for (int t = 1; t < T; ++t)
        if (pthread_create(&th[t], 0, agg_rows, &jobs[t]) != 0) { agg_rows(&jobs[t]); th[t] = 0; jobs[t].r0 = jobs[t].r1; }
    agg_rows(&jobs[0]);
    for (int t = 1; t < T; ++t)
        if (jobs[t].r0 != jobs[t].r1 || th[t]) pthread_join(th[t], 0);
}

/* out[i,:] = scale_i * sum_{k in row i} x[col[k],:]   (scale_i = inv_deg[i] or 1) ; fp32 */
void oracle_csr_aggregate_f32(const int32_t* rowptr, const int32_t* col, const float* inv_deg,
                              const float* x, float* out, int64_t N, int64_t H) {
    oracle_csr_aggregate_ex_f32(rowptr, col, inv_deg, 0, x, 0, out, N, H);
}
