/* CPU oracle in C of the dot-exponential kernel k(x, y) = exp(<x, y>) -- TEST INFRASTRUCTURE ONLY
 * (tests/dot_exponential_oracle.py builds and loads it).  Not in bruteforce.py: a restated oracle for an extension.
 *
 * Float64, one pass pair over the sources per target row, nothing materialised:
 *   pass 1  m = max_j <x_i, y_j> (row normalisation only; 0 otherwise)
 *   pass 2  acc = sum_j exp(<x_i, y_j> - m) b_j, ksum = sum_j exp(<x_i, y_j> - m)
 * Row normalisation returns acc / ksum: softmax(x y^T) b, finite wherever exp(<x, y>) itself would overflow.  The plain
 * product and density (m = 0) are the literal sums, inf where they overflow float64.  Threads: pthreads over
 * interleaved target rows, one per online core.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <unistd.h>

typedef struct {
    int D, E, normalize_rows, tid, nthreads;
    const double *x, *y, *b;
    double* out;
    int64_t n_rows, M;
} job_t;

static double dot(const double* a, const double* b, int D) {
    double s = 0.0;
    for (int d = 0; d < D; ++d) s += a[d] * b[d];
    return s;
}

static void* worker(void* arg) {
    const job_t* J = (const job_t*)arg;
    const int D = J->D, E = J->E;
    for (int64_t r = J->tid; r < J->n_rows; r += J->nthreads) {
        const double* xr = J->x + r * D;
        double m = 0.0;
        if (J->normalize_rows) {
            m = -INFINITY;
            for (int64_t j = 0; j < J->M; ++j) {
                const double s = dot(xr, J->y + j * D, D);
                if (s > m) m = s;
            }
        }
        double acc[256];
        double ksum = 0.0;
        for (int e = 0; e < E; ++e) acc[e] = 0.0;
        for (int64_t j = 0; j < J->M; ++j) {
            const double k = exp(dot(xr, J->y + j * D, D) - m);
            ksum += k;
            if (J->b) for (int e = 0; e < E; ++e) acc[e] += k * J->b[j * E + e];
            else acc[0] += k;
        }
        for (int e = 0; e < E; ++e) J->out[r * E + e] = J->normalize_rows ? acc[e] / ksum : acc[e];
    }
    return NULL;
}

/* x: (n_rows, D), y: (M, D), b: (M, E) or NULL for density, out: (n_rows, E).  Returns 0, or 1 on bad arguments. */
int kmb_dotexp_oracle_f64(const double* x, const double* y, const double* b, double* out, int64_t n_rows, int64_t M, int D,
                          int E, int normalize_rows) {
    if (D < 1 || E < 1 || E > 256 || M < 1) return 1;
    long nc = sysconf(_SC_NPROCESSORS_ONLN);
    int T = nc < 1 ? 1 : (nc > 256 ? 256 : (int)nc);
    if (T > n_rows) T = n_rows > 0 ? (int)n_rows : 1;
    pthread_t th[256];
    job_t jobs[256];
    for (int t = 0; t < T; ++t) {
        job_t j = {D, E, normalize_rows, t, T, x, y, b, out, n_rows, M};
        jobs[t] = j;
        if (t > 0 && pthread_create(&th[t], NULL, worker, &jobs[t]) != 0) return 2;
    }
    worker(&jobs[0]);
    for (int t = 1; t < T; ++t) pthread_join(th[t], NULL);
    return 0;
}
