/* TEST INFRASTRUCTURE ONLY -- plain-C restatement of sparse GPFQ (the L1 penalty of gpfq_set_l1_penalty), the checker of the
 * library's penalty on whole layers.  The walk is stochastic_oracle.c's (the reference's dtype ladder, quantized_network.py:83-121);
 * the step is
 *   q = 0                                                if nrm < 1e-16
 *   v = w_t if |<Xq_t, u>| < 1e-10 else <Xq_t, u + w X_t> / fl(nrm^2)
 *   tau = lambda / fl(nrm^2);  v' = 0 if |v| <= tau else v - copysign(tau, v)
 *   q = Q(v')   nearest (first minimal index on ties) or, with `stochastic`, stoc_round with r = draw(seed, u0 + j, t)
 * with levels fl(scales[j] * A[k]) when scales are given.
 *
 * Build: gcc -O2 -pthread -fPIC -shared -ffp-contract=off -o libsparse_oracle.so sparse_oracle.c -lm
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define DEAD_NORM 1e-16
#define PERP_DOT 1e-10

uint64_t sp_splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

double sp_draw(uint64_t seed, uint64_t u, uint64_t t) {
    return (double)(sp_splitmix64(sp_splitmix64(seed ^ sp_splitmix64(u)) ^ t) >> 11) * 0x1p-53;
}

double sp_stoc_round(double v, const double *A, int K, double r) {
    if (!(v > A[0])) return A[0];
    if (v >= A[K - 1]) return A[K - 1];
    int k = K - 2;
    while (A[k] > v) --k;
    const double p = (v - A[k]) / (A[k + 1] - A[k]);
    return r < p ? A[k + 1] : A[k];
}

double sp_bit_round(double v, const double *A, int K) {
    double best = A[0], bd = fabs(A[0] - v);
    for (int k = 1; k < K; ++k) {
        const double d = fabs(A[k] - v);
        if (d < bd) { bd = d; best = A[k]; }
    }
    return best;
}

double sp_shrink(double v, double tau) { return fabs(v) <= tau ? 0.0 : v - copysign(tau, v); }

static double row_norm(const float *x, long m) {
    double s = 0.0;
    for (long i = 0; i < m; ++i) s += (double)x[i] * (double)x[i];
    return (double)(float)sqrt(s);
}

static void walk(const float *X, const float *Xq, long N0, long m, const float *w, long ldw, const double *A, int K,
                 const double *norms, uint64_t seed, uint64_t unit, double *q, long ldq, double *u, double lambda, int stochastic) {
    memset(u, 0, sizeof(double) * (size_t)m);
    for (long t = 0; t < N0; ++t) {
        const float *x = X + t * m, *xq = Xq + t * m;
        const float wt = w[t * ldw];
        const double r = sp_draw(seed, unit, (uint64_t)t);
        double qt;
        if (norms[t] < DEAD_NORM) {
            qt = 0.0;
        } else {
            double d = 0.0;
            for (long i = 0; i < m; ++i) d += (double)xq[i] * u[i];
            const double den = norms[t] * norms[t];
            double v = (double)wt;
            if (!(fabs(d) < PERP_DOT)) {
                double s = 0.0;
                for (long i = 0; i < m; ++i) {
                    float wx = wt * x[i];
                    s += (double)xq[i] * (u[i] + (double)wx);
                }
                v = s / den;
            }
            v = sp_shrink(v, lambda / den);
            qt = stochastic ? sp_stoc_round(v, A, K, r) : sp_bit_round(v, A, K);
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
    int K, stochastic;
    uint64_t seed;
    double lambda;
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
             jb->ldq, u, jb->lambda, jb->stochastic);
    }
    free(u);
    return NULL;
}

/* Columns j0..j1-1 of a (N0, N1) layer (row stride ldw), unit id u0 + j; scales (nullable) indexed by j; penalty lambda. */
int sp_layer(const float *X, const float *Xq, long N0, long m, const float *W, long ldw, long j0, long j1, const double *alphabet,
             int K, const double *scales, double lambda, int stochastic, uint64_t seed, long u0, double *Q, long ldq, int nthreads) {
    if (N0 <= 0 || m < 0 || K <= 0 || K > 64 || j1 < j0) return 1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    double *norms = (double *)malloc(sizeof(double) * (size_t)N0);
    if (!norms) return 2;
    for (long t = 0; t < N0; ++t) norms[t] = row_norm(Xq + t * m, m);
    long next = j0;
    int fail = 0;
    job_t jb = {X, Xq, W, N0, m, ldw, j1, ldq, u0, alphabet, scales, norms, K, stochastic, seed, lambda, Q, &next, &fail};
    pthread_t th[256];
    int started = 0;
    for (int i = 0; i < nthreads - 1; ++i)
        if (pthread_create(&th[started], NULL, worker, &jb) == 0) ++started;
    worker(&jb);
    for (int i = 0; i < started; ++i) pthread_join(th[i], NULL);
    free(norms);
    return fail ? 2 : 0;
}
