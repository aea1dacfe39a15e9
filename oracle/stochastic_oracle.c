/* TEST INFRASTRUCTURE ONLY -- plain-C restatement of the stochastic-rounding (SPFQ) walk, the checker of the library's
 * GPFQ_ROUND_STOCHASTIC mode.  The walk is gpfq_oracle.c's (the reference's dtype ladder, quantized_network.py:83-121: w*X_t
 * rounded to fp32 per element, q*Xq_t and all sums in fp64, ||Xq_t|| rounded to fp32 and squared in fp64); only the quantizer
 * differs:
 *   splitmix64(x)       = the SplitMix64 finaliser of x + 0x9E3779B97F4A7C15 (mod 2^64)
 *   draw(seed, u, t)    = (splitmix64(splitmix64(seed ^ splitmix64(u)) ^ t) >> 11) * 2^-53
 *   stoc_round(v, A, r) = A[0] unless v > A[0]; A[K-1] if v >= A[K-1]; else with k = max{i : A[i] <= v},
 *                         p = (v - A[k]) / (A[k+1] - A[k]): A[k+1] if r < p else A[k]
 * One step: the literal 0 for a dead direction, stoc_round(w_t) when |<Xq_t, u>| < 1e-10, else stoc_round(<Xq_t, u + w X_t> / nrm^2),
 * with r = draw(seed, u0 + j, t) for column j and levels fl(scales[j] * A[k]) when scales are given.
 *
 * Build: gcc -O2 -pthread -fPIC -shared -ffp-contract=off -o libstochastic_oracle.so stochastic_oracle.c -lm
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define DEAD_NORM 1e-16
#define PERP_DOT 1e-10

uint64_t so_splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

double so_draw(uint64_t seed, uint64_t u, uint64_t t) {
    return (double)(so_splitmix64(so_splitmix64(seed ^ so_splitmix64(u)) ^ t) >> 11) * 0x1p-53;
}

double so_stoc_round(double v, const double *A, int K, double r) {
    if (!(v > A[0])) return A[0];
    if (v >= A[K - 1]) return A[K - 1];
    int k = K - 2;
    while (A[k] > v) --k;
    const double p = (v - A[k]) / (A[k + 1] - A[k]);
    return r < p ? A[k + 1] : A[k];
}

static double row_norm(const float *x, long m) {
    double s = 0.0;
    for (long i = 0; i < m; ++i) s += (double)x[i] * (double)x[i];
    return (double)(float)sqrt(s);
}

static void walk(const float *X, const float *Xq, long N0, long m, const float *w, long ldw, const double *A, int K,
                 const double *norms, uint64_t seed, uint64_t unit, double *q, long ldq, double *u) {
    memset(u, 0, sizeof(double) * (size_t)m);
    for (long t = 0; t < N0; ++t) {
        const float *x = X + t * m, *xq = Xq + t * m;
        const float wt = w[t * ldw];
        const double r = so_draw(seed, unit, (uint64_t)t);
        double qt;
        if (norms[t] < DEAD_NORM) {
            qt = 0.0;
        } else {
            double d = 0.0;
            for (long i = 0; i < m; ++i) d += (double)xq[i] * u[i];
            if (fabs(d) < PERP_DOT) {
                qt = so_stoc_round((double)wt, A, K, r);
            } else {
                double s = 0.0;
                for (long i = 0; i < m; ++i) {
                    float wx = wt * x[i];
                    s += (double)xq[i] * (u[i] + (double)wx);
                }
                qt = so_stoc_round(s / (norms[t] * norms[t]), A, K, r);
            }
        }
        q[t * ldq] = qt;
        for (long i = 0; i < m; ++i) {
            float wx = wt * x[i];
            double qx = qt * (double)xq[i];
            double diff = (double)wx - qx;
            u[i] += diff;
        }
    }
}

typedef struct {
    const float *X, *Xq, *W;
    long N0, m, ldw, j1, ldq, u0;
    const double *alphabet, *scales, *norms;
    int K;
    uint64_t seed;
    double *Q;
    long *next;
    int *fail;
} job_t;

static void *worker(void *arg) {
    job_t *jb = (job_t *)arg;
    double *u = (double *)malloc(sizeof(double) * (size_t)(jb->m > 0 ? jb->m : 1));
    double lev[64];
    if (!u) { __atomic_store_n(jb->fail, 1, __ATOMIC_RELAXED); return NULL; }
    for (;;) {
        long j = __atomic_fetch_add(jb->next, 1, __ATOMIC_RELAXED);
        if (j >= jb->j1) break;
        const double *A = jb->alphabet;
        if (jb->scales) {
            for (int k = 0; k < jb->K; ++k) lev[k] = jb->scales[j] * jb->alphabet[k];
            A = lev;
        }
        walk(jb->X, jb->Xq, jb->N0, jb->m, jb->W + j, jb->ldw, A, jb->K, jb->norms, jb->seed, (uint64_t)(jb->u0 + j), jb->Q + j,
             jb->ldq, u);
    }
    free(u);
    return NULL;
}

/* Columns j0..j1-1 of a (N0, N1) layer (row stride ldw), unit id u0 + j; scales (nullable) indexed by j. */
int so_layer(const float *X, const float *Xq, long N0, long m, const float *W, long ldw, long j0, long j1, const double *alphabet,
             int K, const double *scales, uint64_t seed, long u0, double *Q, long ldq, int nthreads) {
    if (N0 <= 0 || m < 0 || K <= 0 || K > 64 || j1 < j0) return 1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    double *norms = (double *)malloc(sizeof(double) * (size_t)N0);
    if (!norms) return 2;
    for (long t = 0; t < N0; ++t) norms[t] = row_norm(Xq + t * m, m);
    long next = j0;
    int fail = 0;
    job_t jb = {X, Xq, W, N0, m, ldw, j1, ldq, u0, alphabet, scales, norms, K, seed, Q, &next, &fail};
    pthread_t th[256];
    int started = 0;
    for (int i = 0; i < nthreads - 1; ++i)
        if (pthread_create(&th[started], NULL, worker, &jb) == 0) ++started;
    worker(&jb);
    for (int i = 0; i < started; ++i) pthread_join(th[i], NULL);
    free(norms);
    return fail ? 2 : 0;
}
