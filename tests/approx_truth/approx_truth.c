/* Ground truth of approximate search, for the tests of kmer_b200_search_approx_batch (not the reference, which has no
   such function): per query q of length m, sorted { p : p + m <= n, Hamming(T[p, p+m), q) <= e } by a scan of every
   window with an early exit once a window has more than e mismatches. The queries are shared out over n_threads
   threads; each thread collects its queries' positions in order and the lists are concatenated. */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    const uint8_t *text, *q;
    const uint64_t *q_off;
    uint64_t n, lo, hi, *counts;
    uint32_t e;
    uint32_t *pos;
    uint64_t n_pos, cap_pos;
} approx_job;

static void *approx_worker(void *arg)
{
    approx_job *j = (approx_job *)arg;
    for (uint64_t i = j->lo; i < j->hi; ++i) {
        const uint8_t *qq = j->q + j->q_off[i];
        const uint64_t m = j->q_off[i + 1] - j->q_off[i];
        uint64_t c = 0;
        if (m > 0 && m <= j->n) {
            for (uint64_t p = 0; p + m <= j->n; ++p) {
                const uint8_t *t = j->text + p;
                uint32_t d = 0;
                for (uint64_t s = 0; s < m && d <= j->e; ++s)
                    d += t[s] != qq[s];
                if (d > j->e)
                    continue;
                if (j->n_pos == j->cap_pos) {
                    j->cap_pos = j->cap_pos ? 2 * j->cap_pos : 1024;
                    j->pos = (uint32_t *)realloc(j->pos, j->cap_pos * sizeof(uint32_t));
                }
                j->pos[j->n_pos++] = (uint32_t)p;
                ++c;
            }
        }
        j->counts[i] = c;
    }
    return NULL;
}

/* counts[Q]; *positions (malloc'ed, free with approx_truth_free) holds *total positions, query by query */
int approx_truth_batch(const uint8_t *text, uint64_t n, const uint8_t *q, const uint64_t *q_off, uint64_t Q, uint32_t e,
                       uint32_t n_threads, uint64_t *counts, uint32_t **positions, uint64_t *total)
{
    if (n_threads == 0)
        n_threads = 1;
    if (n_threads > 256)
        n_threads = 256;
    approx_job jobs[256];
    pthread_t th[256];
    for (uint32_t t = 0; t < n_threads; ++t) {
        memset(&jobs[t], 0, sizeof(approx_job));
        jobs[t].text = text;
        jobs[t].n = n;
        jobs[t].q = q;
        jobs[t].q_off = q_off;
        jobs[t].lo = Q * t / n_threads;
        jobs[t].hi = Q * (t + 1) / n_threads;
        jobs[t].counts = counts;
        jobs[t].e = e;
        pthread_create(&th[t], NULL, approx_worker, &jobs[t]);
    }
    uint64_t tot = 0;
    for (uint32_t t = 0; t < n_threads; ++t) {
        pthread_join(th[t], NULL);
        tot += jobs[t].n_pos;
    }
    *total = tot;
    *positions = (uint32_t *)malloc((tot ? tot : 1) * sizeof(uint32_t));
    uint64_t o = 0;
    for (uint32_t t = 0; t < n_threads; ++t) {
        if (jobs[t].n_pos)
            memcpy(*positions + o, jobs[t].pos, jobs[t].n_pos * sizeof(uint32_t));
        o += jobs[t].n_pos;
        free(jobs[t].pos);
    }
    return 0;
}

void approx_truth_free(void *p)
{
    free(p);
}
