// gmm.cu -- the class model of the pipeline on the device: StandardScaler + full-covariance Gaussian mixture (EM).
//
// Replaces the host round trip of imsegm/graph_cuts.py:73-163 (estim_class_model, default 'GMM'):
//   sklearn Pipeline[StandardScaler, GaussianMixture(n_components=K, covariance_type='full',
//                                                    n_init=int(sqrt(max_iter)), max_iter=max_iter)]
//   followed by predict_proba (imsegm/pipelines.py:95-96).
// The EM restates sklearn.mixture.GaussianMixture (tol 1e-3 on the mean log-likelihood, reg_covar 1e-6,
// weights = (sum resp + 10 eps) / N, centred covariance, precision Cholesky, best of n_init by lower bound).
// Each of the n_init restarts runs in its own CTA, all restarts concurrently; the initial hard assignment is
// either supplied (init_labels: makes the fit deterministic and comparable with sklearn from the same start) or
// k-means++ / Lloyd with a counter-based RNG (the reference leaves the model unseeded, so only the algorithm,
// not a label-for-label result, can be matched; tests compare against sklearn from a shared initialisation).
// N is tiny (superpixels, not pixels): this stage is latency bound, it exists to remove the host sync.
#include "common.cuh"
#include <float.h>
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace {

constexpr int GT = 512;      // threads per restart CTA
constexpr int DMAX = 16;     // feature dimensions of the single-kernel path (one CTA per restart, everything on chip)
constexpr int CLI = 8;       // CTAs per restart (one thread-block cluster) in the large-D initialisation
constexpr int KS = 8;        // split-K factor of the M-step Gram matrices
constexpr int DBIG = 232;    // feature dimensions of the large-D path (batched GEMMs, e.g. colour + Leung-Malik = 189); the packed
                             // lower triangle of one covariance (D (D + 1) / 2 doubles) has to fit the shared memory of a CTA
constexpr int KMAX = 8;      // mixture components handled on the device

struct GmmWs {
    double* xs;       // [N, D] standardised features
    double* scale;    // [2 D] mean, scale
    double* resp;     // [n_init, N, K]
    int* lab;         // [n_init, N]
    double* par;      // [n_init, PSTRIDE]: weights K | means K D | cov K D D | prec_chol K D D | lower_bound | n_iter | converged | ok
    double* red;      // [n_init, GT] scratch
    // large-D path only (D > DMAX)
    double* big;      // [n_init, K, N, D]  Y = X U (E-step) / sqrt(r) (X - mu) (M-step); never live at the same time
    double* bvec;     // [n_init, K, D]     mu U
    double* ldw;      // [n_init, K]        log|prec_chol| + log weight
    double* lowpart;  // [n_init, ceil(N / 8)] per-block sums of the log-likelihood
    double* cent;     // [n_init, 2, K, D]  k-means centres (double buffered)
    int* iflag;       // [n_init, CLI]      "a label changed" per CTA of the init cluster
    double* gram;     // [n_init, K, KS, D, D] split-K partial Gram matrices of the M-step
    double* sresp;    // [n_init, N, K]     sqrt(resp), the weights of the M-step Gram matrices
    double* tot;      // [n_init, K, 1 + D] k-means counts / coordinate sums
    double* state;    // [n_init, 4]        lower bound of the previous E-step, done, -, failed
    int* flag;        // [1]                restarts still running
};

__host__ __device__ inline int pstride(int K, int D) { return K + K * D + 2 * K * D * D + 4; }

struct Rng {
    unsigned long long s;
    __device__ explicit Rng(unsigned long long seed) : s(seed) {}
    __device__ unsigned long long next()
    {
        unsigned long long z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    __device__ double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
};

__device__ double block_sum_d(double v, double* s_red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0;
    for (int i = 0; i < GT / 32; ++i) t += s_red[i];
    return t;
}

// StandardScaler: mean / population std per feature (zero variance -> scale 1), one CTA per feature
__global__ void __launch_bounds__(GT) k_gmm_scale(const double* __restrict__ feat, int N_in, const int* n_dev, int D, int ld, int use_scaler,
                                                  GmmWs w)
{
    __shared__ double s_red[GT / 32];
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    {
        const int d = blockIdx.x;
        double s = 0;
        for (int n = threadIdx.x; n < N; n += GT) s += feat[(size_t)n * ld + d];
        double mean = block_sum_d(s, s_red) / N;
        double v = 0;
        for (int n = threadIdx.x; n < N; n += GT) { double t = feat[(size_t)n * ld + d] - mean; v += t * t; }
        double var = block_sum_d(v, s_red) / N;
        double sc = sqrt(var);
        // sklearn _is_constant_feature: var <= N eps var + (N mean eps)^2  -> scale 1
        const double ub = N * DBL_EPSILON * var + (N * mean * DBL_EPSILON) * (N * mean * DBL_EPSILON);
        if (var <= ub) sc = 1.0;
        if (!use_scaler) { mean = 0.0; sc = 1.0; }
        if (threadIdx.x == 0) { w.scale[d] = mean; w.scale[D + d] = sc; }
        for (int n = threadIdx.x; n < N; n += GT) w.xs[(size_t)n * D + d] = (feat[(size_t)n * ld + d] - mean) / sc;
        __syncthreads();
    }
}

// log N(x | mu_k, prec_chol_k) for all k; returns log-sum-exp of (log w_k + log N_k), fills lw[k] with the terms
__device__ __forceinline__ double log_prob_all(const double* x, int D, int K, const double* wts, const double* mu, const double* pc,
                                               const double* logdet, double* lw)
{
    double mx = -DBL_MAX;
    for (int k = 0; k < K; ++k) {
        const double* m = mu + k * D;
        const double* U = pc + (size_t)k * D * D; // upper triangular: y_j = sum_{i<=j} (x_i - m_i) U[i][j]
        double q = 0;
        for (int j = 0; j < D; ++j) {
            double y = 0;
            for (int i = 0; i <= j; ++i) y += (x[i] - m[i]) * U[i * D + j];
            q += y * y;
        }
        double lp = -0.5 * (D * 1.8378770664093453 + q) + logdet[k]; // logdet[k] already holds log|prec_chol_k| + log w_k
        lw[k] = lp;
        mx = fmax(mx, lp);
    }
    double s = 0;
    for (int k = 0; k < K; ++k) s += exp(lw[k] - mx);
    return mx + log(s);
}

// ---- the single-kernel path (D <= DMAX): one thread-block CLUSTER of CL CTAs per restart ------------------------------------------
// The samples of a restart are cut into CL contiguous ranges, one per CTA of the cluster.  Every CTA keeps a bit-identical replica of
// the model parameters in its shared memory; what crosses the CTAs are the partial sums of the reductions (log-likelihood, component
// weights / means / covariances, k-means counts), exchanged through distributed shared memory and added in rank order by every CTA,
// so the replicas never diverge.  CL = 1 is the plain one-CTA-per-restart kernel (small N).

struct ClusterCtx {
    int rank, CL;
    double* s_x;      // [GT] exchange buffer of this CTA (remote CTAs read it through DSMEM)
    double* s_red;    // [GT / 32]
};

// every thread contributes `v`; every thread of every CTA of the cluster gets the same total (partials added in rank order)
__device__ double cluster_sum(double v, const ClusterCtx& c)
{
    const double t = block_sum_d(v, c.s_red);
    if (c.CL == 1) return t;
    cg::cluster_group cl = cg::this_cluster();
    if (threadIdx.x == 0) c.s_x[0] = t;
    cl.sync();
    double tot = 0;
    for (int r = 0; r < c.CL; ++r) tot += *cl.map_shared_rank(&c.s_x[0], r);
    cl.sync();
    return tot;
}

// threads [0, nq) hold one partial each (their quantity's sum over this CTA's samples); returns the cluster-wide sum of the
// thread's quantity (partials added in rank order).  Collective: every thread of every CTA must call it.
__device__ double cluster_vec_sum(double part, int nq, const ClusterCtx& c)
{
    if (c.CL == 1) return part;
    cg::cluster_group cl = cg::this_cluster();
    if ((int)threadIdx.x < nq) c.s_x[threadIdx.x] = part;
    cl.sync();
    double tot = 0;
    if ((int)threadIdx.x < nq)
        for (int r = 0; r < c.CL; ++r) tot += *cl.map_shared_rank(&c.s_x[threadIdx.x], r);
    cl.sync();
    return tot;
}

// parameters from responsibilities (sklearn _estimate_gaussian_parameters + _compute_precision_cholesky) over the samples
// [n_lo, n_hi) of this CTA, merged over the cluster; `par` is this CTA's shared-memory replica.
// returns false when a covariance is not positive definite (the same answer in every CTA)
__device__ bool m_step(const double* __restrict__ xs, const double* __restrict__ resp, int n_lo, int n_hi, int N, int D, int K, double reg,
                       double* par, double* s_part, const ClusterCtx& c)
{
    double* wts = par; double* mu = par + K; double* cov = mu + K * D; double* pc = cov + (size_t)K * D * D;
    // pass 1: nk and means, quantity-parallel over sample slices
    const int Q1 = K * (1 + D);
    for (int q0 = 0; q0 < Q1; q0 += GT) {
        const int nq = min(GT, Q1 - q0);
        const int S = max(1, GT / nq);
        const int q = q0 + (threadIdx.x % nq), sl = threadIdx.x / nq;
        double acc = 0;
        if (sl < S) {
            const int k = q / (1 + D), j = q % (1 + D);
            for (int n = n_lo + sl; n < n_hi; n += S) {
                double r = resp[(size_t)n * K + k];
                acc += j == 0 ? r : r * xs[(size_t)n * D + j - 1];
            }
        }
        s_part[threadIdx.x] = acc;
        __syncthreads();
        double t = 0;
        if ((int)threadIdx.x < nq)
            for (int s2 = 0; s2 < S; ++s2) t += s_part[s2 * nq + threadIdx.x];
        t = cluster_vec_sum(t, nq, c);
        if ((int)threadIdx.x < nq) {
            const int k = q / (1 + D), j = q % (1 + D);
            if (j == 0) wts[k] = t + 10 * DBL_EPSILON; // nk (divided by N at the end)
            else mu[k * D + j - 1] = t;                 // sum r x (divided by nk below)
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < K * D; i += GT) mu[i] = mu[i] / wts[i / D];
    __syncthreads();
    // pass 2: centred covariances (upper triangle), quantity-parallel
    const int T = D * (D + 1) / 2, Q2 = K * T;
    for (int q0 = 0; q0 < Q2; q0 += GT) {
        const int nq = min(GT, Q2 - q0);
        const int S = max(1, GT / nq);
        const int q = q0 + (threadIdx.x % nq), sl = threadIdx.x / nq;
        int k = q / T, t = q % T, a = 0;
        while (t >= D - a) { t -= D - a; ++a; }
        const int b = a + t; // (a, b), a <= b
        double acc = 0;
        if (sl < S) {
            const double ma = mu[k * D + a], mb = mu[k * D + b];
            for (int n = n_lo + sl; n < n_hi; n += S)
                acc += resp[(size_t)n * K + k] * (xs[(size_t)n * D + a] - ma) * (xs[(size_t)n * D + b] - mb);
        }
        s_part[threadIdx.x] = acc;
        __syncthreads();
        double tt = 0;
        if ((int)threadIdx.x < nq)
            for (int s2 = 0; s2 < S; ++s2) tt += s_part[s2 * nq + threadIdx.x];
        tt = cluster_vec_sum(tt, nq, c);
        if ((int)threadIdx.x < nq) {
            double cc = tt / wts[k] + (a == b ? reg : 0.0);
            cov[(size_t)k * D * D + a * D + b] = cc;
            cov[(size_t)k * D * D + b * D + a] = cc;
        }
        __syncthreads();
    }
    // Cholesky cov = L L^T, prec_chol = (L^-1)^T, one thread per component
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    if (threadIdx.x < K) {
        const int k = threadIdx.x;
        const double* Cm = cov + (size_t)k * D * D;
        double* U = pc + (size_t)k * D * D;
        double L[DMAX * DMAX];
        bool ok = true;
        for (int i = 0; i < D && ok; ++i)
            for (int j = 0; j <= i; ++j) {
                double s = Cm[i * D + j];
                for (int p = 0; p < j; ++p) s -= L[i * D + p] * L[j * D + p];
                if (i == j) { if (!(s > 0)) { ok = false; break; } L[i * D + i] = sqrt(s); }
                else L[i * D + j] = s / L[j * D + j];
            }
        if (!ok) s_bad = 1;
        else {
            // Z = L^-1 (lower);  U = Z^T
            for (int cc = 0; cc < D; ++cc)
                for (int r = 0; r < D; ++r) {
                    if (r < cc) { U[cc * D + r] = 0.0; continue; }
                    double s = (r == cc) ? 1.0 : 0.0;
                    for (int p = cc; p < r; ++p) s -= L[r * D + p] * U[cc * D + p]; // U[cc][p] holds Z[p][cc]
                    U[cc * D + r] = s / L[r * D + r];
                }
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += GT) wts[k] = wts[k] / N;
    __syncthreads();
    return s_bad == 0;
}

// one cluster of CL CTAs per restart (gridDim.x = n_init * CL, cluster dimension CL set at launch)
__global__ void __launch_bounds__(GT) k_gmm_fit(int N_in, const int* n_dev, int D, int K, int max_iter, double tol, double reg,
                                               unsigned long long seed, const int* __restrict__ init_labels, int CL, GmmWs w)
{
    extern __shared__ double s_dyn[];          // parameter replica [pstride(K, D)]
    __shared__ double s_part[GT];
    __shared__ double s_x[GT];
    __shared__ double s_red[GT / 32];
    __shared__ double s_logdet[KMAX];
    __shared__ double s_cent[KMAX * DMAX];
    __shared__ double s_tot[KMAX * (1 + DMAX)];
    __shared__ int s_pick;
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int init = blockIdx.x / CL;
    ClusterCtx c;
    c.rank = blockIdx.x % CL; c.CL = CL; c.s_x = s_x; c.s_red = s_red;
    const int chunk_n = (N + CL - 1) / CL;
    const int n_lo = min(N, c.rank * chunk_n), n_hi = min(N, n_lo + chunk_n);   // the samples of this CTA
    const double* xs = w.xs;
    double* resp = w.resp + (size_t)init * N_in * K;
    int* lab = w.lab + (size_t)init * N_in;
    double* par = s_dyn;
    double* gpar = w.par + (size_t)init * pstride(K, D);
    double* wts = par; double* mu = par + K; double* pc = mu + K * D + (size_t)K * D * D;

    // ---- initial hard assignment ----
    if (init_labels) {
        for (int n = n_lo + threadIdx.x; n < n_hi; n += GT) lab[n] = init_labels[(size_t)init * N_in + n];
        __syncthreads();
    } else {
        // k-means++ seeding (one D^2-weighted draw per centre), then Lloyd
        Rng rng(seed * 0x100000001B3ull + 1469598103934665603ull * (unsigned long long)(init + 1));
        double* d2 = w.red + (size_t)init * N_in; // closest squared distance per sample
        int first = (int)(rng.uniform() * N); if (first >= N) first = N - 1;
        for (int d = threadIdx.x; d < D; d += GT) s_cent[d] = xs[(size_t)first * D + d];
        __syncthreads();
        for (int cc = 1; cc <= K; ++cc) {
            // update closest distances with centre cc-1
            double loc = 0;
            for (int n = n_lo + threadIdx.x; n < n_hi; n += GT) {
                double s = 0;
                for (int d = 0; d < D; ++d) { double t = xs[(size_t)n * D + d] - s_cent[(cc - 1) * D + d]; s += t * t; }
                double cur = (cc == 1) ? s : fmin(d2[n], s);
                d2[n] = cur;
                loc += cur;
            }
            // total over the cluster AND the running sum of the ranks before this one (the draw walks the samples in order)
            const double mine = block_sum_d(loc, s_red);
            double total = mine, before = 0;
            if (CL > 1) {
                cg::cluster_group cl = cg::this_cluster();
                if (threadIdx.x == 0) s_x[0] = mine;
                cl.sync();
                total = 0;
                for (int r = 0; r < CL; ++r) { const double pr = *cl.map_shared_rank(&s_x[0], r); if (r < c.rank) before += pr; total += pr; }
                cl.sync();
            }
            if (cc == K) break;
            const double thr = rng.uniform() * total; // same on every thread of every CTA (same rng state)
            // the CTA whose range holds thr: contiguous per-thread chunks -> prefix over chunk sums -> the chunk holding thr scans itself
            const bool holder = (thr > before || c.rank == 0) && (thr <= before + mine || c.rank == CL - 1);
            const int nloc = n_hi - n_lo;
            const int chunk = (nloc + GT - 1) / GT, beg = n_lo + threadIdx.x * chunk, end = min(beg + chunk, n_hi);
            double cs = 0;
            for (int n = beg; n < end; ++n) cs += d2[n];
            s_part[threadIdx.x] = cs;
            if (threadIdx.x == 0) s_pick = -1;
            __syncthreads();
            if (threadIdx.x == 0 && holder && nloc > 0) {
                double run = before; int t = 0;
                for (; t < GT; ++t) { if (run + s_part[t] >= thr) break; run += s_part[t]; }
                int pick = n_hi - 1;
                if (t < GT) {
                    int b2 = n_lo + t * chunk, e2 = min(b2 + chunk, n_hi), n = b2;
                    for (; n < e2; ++n) { run += d2[n]; if (run >= thr) break; }
                    pick = min(n, n_hi - 1);
                }
                s_pick = pick;
            }
            __syncthreads();
            // the lowest-ranked CTA that made a pick publishes it (rounding may make two neighbours claim the threshold)
            int pick = s_pick;
            if (CL > 1) {
                cg::cluster_group cl = cg::this_cluster();
                if (threadIdx.x == 0) s_x[1] = (double)s_pick;
                cl.sync();
                pick = -1;
                for (int r = 0; r < CL && pick < 0; ++r) pick = (int)*cl.map_shared_rank(&s_x[1], r);
                cl.sync();
            }
            if (pick < 0) pick = N - 1;
            for (int d = threadIdx.x; d < D; d += GT) s_cent[cc * D + d] = xs[(size_t)pick * D + d];
            __syncthreads();
        }
        // Lloyd iterations (sklearn KMeans: max_iter 300, tol 1e-4 * mean feature variance; X is standardised)
        for (int n = n_lo + threadIdx.x; n < n_hi; n += GT) lab[n] = -1;
        for (int it = 0; it < 300; ++it) {
            int changed = 0;
            for (int n = n_lo + threadIdx.x; n < n_hi; n += GT) {
                double best = DBL_MAX; int bk = 0;
                for (int k = 0; k < K; ++k) {
                    double s = 0;
                    for (int d = 0; d < D; ++d) { double t = xs[(size_t)n * D + d] - s_cent[k * D + d]; s += t * t; }
                    if (s < best) { best = s; bk = k; }
                }
                if (lab[n] != bk) { lab[n] = bk; changed = 1; }
            }
            // new centres: count and coordinate sums of every cluster in ONE quantity-parallel pass over sample slices
            // (quantity q = (k, j): j == 0 the count, j >= 1 the sum of coordinate j-1); quantity Q carries the "changed" flag
            const int Q = K * (1 + D);                 // <= 8 * 17 = 136 < GT
            const int S = max(1, GT / (Q + 1));
            {
                const int q = threadIdx.x % (Q + 1), sl = threadIdx.x / (Q + 1);
                double a = 0;
                if (sl < S && q < Q) {
                    const int k = q / (1 + D), j = q % (1 + D);
                    for (int n = n_lo + sl; n < n_hi; n += S)
                        if (lab[n] == k) a += j == 0 ? 1.0 : xs[(size_t)n * D + j - 1];
                }
                s_part[threadIdx.x] = a;
            }
            changed = __syncthreads_or(changed);
            double t = 0;
            if ((int)threadIdx.x < Q) { for (int s2 = 0; s2 < S; ++s2) t += s_part[s2 * (Q + 1) + threadIdx.x]; }
            else if ((int)threadIdx.x == Q) t = changed ? 1.0 : 0.0;
            t = cluster_vec_sum(t, Q + 1, c);
            if ((int)threadIdx.x <= Q) s_tot[threadIdx.x] = t;
            __syncthreads();
            changed = s_tot[Q] != 0.0;
            double shift = 0;
            for (int k = 0; k < K; ++k) {
                const double cnt = s_tot[k * (1 + D)];
                if (cnt > 0)
                    for (int d = 0; d < D; ++d) { const double tt = s_tot[k * (1 + D) + 1 + d] / cnt - s_cent[k * D + d]; shift += tt * tt; }
            }
            __syncthreads();
            if ((int)threadIdx.x < K * D) {
                const int k = threadIdx.x / D, d = threadIdx.x % D;
                const double cnt = s_tot[k * (1 + D)];
                if (cnt > 0) s_cent[threadIdx.x] = s_tot[k * (1 + D) + 1 + d] / cnt;
            }
            __syncthreads();
            if (!changed || shift <= 1e-4) break;
        }
        __syncthreads();
    }
    for (int i = n_lo * K + threadIdx.x; i < n_hi * K; i += GT) resp[i] = (lab[i / K] == i % K) ? 1.0 : 0.0;
    __syncthreads();

    // ---- EM ----
    bool ok = m_step(xs, resp, n_lo, n_hi, N, D, K, reg, par, s_part, c);
    double lower = -DBL_MAX;
    int it = 0, conv = 0;
    if (ok) {
        for (it = 1; it <= max_iter; ++it) {
            const double prev = lower;
            if (threadIdx.x < K) {
                double ld = 0;
                for (int j = 0; j < D; ++j) ld += log(pc[(size_t)threadIdx.x * D * D + j * D + j]);
                s_logdet[threadIdx.x] = ld + log(wts[threadIdx.x]);
            }
            __syncthreads();
            double acc = 0;
            for (int n = n_lo + threadIdx.x; n < n_hi; n += GT) {
                double lw[KMAX];
                double lse = log_prob_all(xs + (size_t)n * D, D, K, wts, mu, pc, s_logdet, lw);
                for (int k = 0; k < K; ++k) resp[(size_t)n * K + k] = exp(lw[k] - lse);
                acc += lse;
            }
            lower = cluster_sum(acc, c) / N;
            ok = m_step(xs, resp, n_lo, n_hi, N, D, K, reg, par, s_part, c);
            if (!ok) break;
            if (it > 1 && fabs(lower - prev) < tol) { conv = 1; break; }
        }
        if (it > max_iter) it = max_iter;
    }
    // rank 0 publishes the replica (every replica is identical) and the outcome of the restart
    if (c.rank == 0) {
        const int np = K + K * D + 2 * K * D * D;
        for (int i = threadIdx.x; i < np; i += GT) gpar[i] = par[i];
        if (threadIdx.x == 0) {
            double* tail = gpar + np; // lower_bound, n_iter, converged, ok
            tail[0] = ok ? lower : -DBL_MAX; tail[1] = (double)it; tail[2] = (double)conv; tail[3] = ok ? 1.0 : 0.0;
        }
    }
    if (CL > 1) cg::this_cluster().sync();   // no CTA may exit while a neighbour can still read its exchange buffer
}


// ---------------------------------------------------------------------------------------------------------------------
// Large-D path (DMAX < D <= DBIG), e.g. colour + full Leung-Malik statistics: D = 189 (BASELINE config 3).
// The same EM, restructured around its two contractions, all restarts and components in one launch each:
//   E-step:  Y[r,k] = X U[r,k]                (N x D x D per (restart, component))   -> k_dgemm_batched<false>
//   M-step:  C[r,k] = Xw[r,k]^T Xw[r,k],  Xw = sqrt(resp) (X - mu)   (D x D x N)     -> k_dgemm_batched<true>
// with a CTA-parallel Cholesky / triangular inverse per (r,k) between them.  The host loop runs the restarts in lock step
// and reads one int per iteration (restarts still running); a converged restart is frozen (its CTAs exit at once).
// FP64 throughout (the reference's scikit-learn model is float64); explicit fma() because the file is built with -fmad=false.
// ---------------------------------------------------------------------------------------------------------------------

constexpr int TM = 96, TN = 96, TK = 16;   // CTA tile of the FP64 GEMMs: 256 threads, a 6 x 6 register tile each
constexpr int MT = TM / 16;                // (192 = 2 x 96 covers D = 189 with 3 % padding; six consecutive doubles per operand and k: three 16-byte loads)
constexpr int GQ = TM * TK / 256;          // elements of one operand a thread stages per k-step

// C[b] (M x Nn) = op(A[b]) B[b], row-major; TRANS_A: A[b] is stored Kd x M.  The sample count may come from the device (n_dev).
// Batch b = (restart r, component k) = (b / per, b % per); operand X of the batch starts at X + r * strideXr + k * strideXk.
// A batch whose restart is done is skipped.
struct BatchStride { size_t ar, ak, br, bk, cr, ck, cs; };
// ksplit > 1: the contraction index is cut into ksplit ranges, range s of batch b is blockIdx.z = b * ksplit + s and writes its
// partial product at C + ... + s * cs (the consumer adds the partials in order).  The next tile's global loads are issued before
// the current tile is multiplied.
// FUSE_W (with TRANS_A, the M-step): A and B are both the standardised features X [Kd x D]; element (n, m) is taken as
// sr[n] (X[n][m] - mu[m]) with sr = sqrt(resp) of the batch's (restart, component) -- the weighted, centred copy is never stored.
// b_upper: B[b] is upper triangular, so columns n0.. only need the rows below n0 + TN.
struct FuseW { const double* sresp; const double* mu; size_t sr_r; int K; size_t mu_r; int D; };
template <bool TRANS_A, bool FUSE_W>
__global__ void __launch_bounds__(256, 2) k_dgemm_batched(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb,
                                                       double* __restrict__ C, int ldc, BatchStride bs, int M_in, int Nn, int Kd_in,
                                                       const int* n_dev, int n_is_m, const double* state, int per, int upper_only, int ksplit,
                                                       int b_upper, FuseW fw)
{
    __shared__ __align__(16) double As[TK][TM + 4];
    __shared__ __align__(16) double Bs[TK][TN + 4];
    const int b = blockIdx.z / ksplit, split = blockIdx.z % ksplit, br = b / per, bk = b % per;
    if (state && state[(size_t)br * 4 + 1] != 0.0) return;
    if (upper_only && blockIdx.x < blockIdx.y) return;   // symmetric result: tiles below the diagonal are not needed
    const int nlim = n_dev ? *n_dev : 0x7fffffff;
    const int M = n_is_m ? min(M_in, nlim) : M_in;       // the sample count is M (E-step) or Kd (M-step)
    const int Kd = n_is_m ? Kd_in : min(Kd_in, nlim);
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    if (m0 >= M) return;
    A += br * bs.ar + bk * bs.ak; B += br * bs.br + bk * bs.bk; C += br * bs.cr + bk * bs.ck + split * bs.cs;
    const int tiles = (Kd + TK - 1) / TK, tper = (tiles + ksplit - 1) / ksplit;
    const int k_begin = split * tper * TK;
    int k_end = min(Kd, (split + 1) * tper * TK);
    if (b_upper) k_end = min(k_end, n0 + TN);
    const double* sr = FUSE_W ? fw.sresp + br * fw.sr_r + bk : nullptr;          // sr[n * K]
    const double* mu = FUSE_W ? fw.mu + br * fw.mu_r + (size_t)bk * fw.D : nullptr;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[MT][MT];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < MT; ++j) acc[i][j] = 0.0;
    double ra[GQ], rb[GQ];
    auto gload = [&](int k0) {
#pragma unroll
        for (int q = 0; q < GQ; ++q) {
            const int i = threadIdx.x + q * 256;
            int kk, mm;
            if (TRANS_A) { kk = i / TM; mm = i % TM; } else { mm = i / TK; kk = i % TK; }
            const int gm = m0 + mm, gk = k0 + kk;
            ra[q] = (gm < M && gk < k_end) ? (TRANS_A ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk]) : 0.0;
            const int kb = i / TN, nn = i % TN;
            const int gkb = k0 + kb, gn = n0 + nn;
            rb[q] = (gkb < k_end && gn < Nn) ? B[(size_t)gkb * ldb + gn] : 0.0;
            if (FUSE_W) {   // TRANS_A: kk == kb (TM == TN), one weight for both operands
                const double wgt = gk < k_end ? sr[(size_t)gk * fw.K] : 0.0;
                ra[q] = (gm < M && gk < k_end) ? wgt * (ra[q] - mu[gm]) : 0.0;
                rb[q] = (gkb < k_end && gn < Nn) ? wgt * (rb[q] - mu[gn]) : 0.0;
            }
        }
    };
    if (k_begin < k_end) gload(k_begin);
    for (int k0 = k_begin; k0 < k_end; k0 += TK) {
#pragma unroll
        for (int q = 0; q < GQ; ++q) {
            const int i = threadIdx.x + q * 256;
            if (TRANS_A) As[i / TM][i % TM] = ra[q]; else As[i % TK][i / TK] = ra[q];
            Bs[i / TN][i % TN] = rb[q];
        }
        __syncthreads();
        if (k0 + TK < k_end) gload(k0 + TK);
#pragma unroll
        for (int kk = 0; kk < TK; ++kk) {
            double a[MT], bb[MT];
#pragma unroll
            for (int i = 0; i < MT; ++i) { a[i] = As[kk][ty * MT + i]; bb[i] = Bs[kk][tx * MT + i]; }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < MT; ++j) acc[i][j] = fma(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < MT; ++i) {
        const int gm = m0 + ty * MT + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < MT; ++j) {
            const int gn = n0 + tx * MT + j;
            if (gn < Nn) C[(size_t)gm * ldc + gn] = acc[i][j];
        }
    }
}

// StandardScaler for many features: one CTA per 32 features, warps over the samples, lanes over the features; per-warp partials
// are added in warp order (k_gmm_scale walks the features one by one -- fine for D <= 16, 2.4 ms at D = 189)
__global__ void __launch_bounds__(1024) k_big_scale(const double* __restrict__ feat, int N_in, const int* n_dev, int D, int ld, int use_scaler,
                                                   GmmWs w)
{
    __shared__ double s_acc[32][33];
    __shared__ double s_mean[32], s_scale[32];
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int d = blockIdx.x * 32 + lane;
    double a = 0;
    if (d < D) for (int n = wid; n < N; n += 32) a += feat[(size_t)n * ld + d];
    s_acc[wid][lane] = a;
    __syncthreads();
    if (wid == 0) { double t = 0; for (int i = 0; i < 32; ++i) t += s_acc[i][lane]; s_mean[lane] = t / N; }
    __syncthreads();
    const double mean = s_mean[lane];
    a = 0;
    if (d < D) for (int n = wid; n < N; n += 32) { const double t = feat[(size_t)n * ld + d] - mean; a = fma(t, t, a); }
    s_acc[wid][lane] = a;
    __syncthreads();
    if (wid == 0) {
        double t = 0;
        for (int i = 0; i < 32; ++i) t += s_acc[i][lane];
        const double var = t / N;
        double sc = sqrt(var), mu = mean;
        const double ub = N * DBL_EPSILON * var + (N * mean * DBL_EPSILON) * (N * mean * DBL_EPSILON); // sklearn _is_constant_feature
        if (var <= ub) sc = 1.0;
        if (!use_scaler) { mu = 0.0; sc = 1.0; }
        s_mean[lane] = mu; s_scale[lane] = sc;
        if (d < D) { w.scale[d] = mu; w.scale[D + d] = sc; }
    }
    __syncthreads();
    if (d < D) {
        const double mu = s_mean[lane], sc = s_scale[lane];
        for (int n = wid; n < N; n += 32) w.xs[(size_t)n * D + d] = (feat[(size_t)n * ld + d] - mu) / sc;
    }
}

// initial hard assignment of every restart: supplied labels, or k-means++ / Lloyd as in k_gmm_fit.  One thread-block cluster of
// CLI CTAs per restart; samples are spread over all warps of the cluster, the state (centres, labels, sums) lives in global
// memory and cluster.sync() orders it.  Every CTA draws the same random numbers, so the control flow is identical in all of them.
__global__ void __cluster_dims__(CLI, 1, 1) __launch_bounds__(GT) k_big_init(int N_in, const int* n_dev, int D, int K, unsigned long long seed,
                                                                          const int* __restrict__ init_labels, GmmWs w)
{
    cg::cluster_group cl = cg::this_cluster();
    __shared__ double s_part[GT];
    __shared__ double s_red[GT / 32];
    __shared__ double s_acc[GT / 32][33];
    __shared__ int s_pick;
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int init = blockIdx.x / CLI, rank = (int)cl.block_rank();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = GT / 32;
    const int gw = rank * nw + wid, gnw = CLI * nw;          // warp index / warp count inside the restart
    const int gt = rank * GT + threadIdx.x, gnt = CLI * GT;  // thread index / thread count inside the restart
    const double* xs = w.xs;
    double* resp = w.resp + (size_t)init * N_in * K;
    int* lab = w.lab + (size_t)init * N_in;
    double* cent = w.cent + (size_t)init * 2 * K * D;
    double* tot = w.tot + (size_t)init * K * (1 + D);
    int* chg = w.iflag + init * CLI;
    if (gt == 0) { w.state[init * 4] = -DBL_MAX; w.state[init * 4 + 1] = 0.0; w.state[init * 4 + 2] = 0.0; w.state[init * 4 + 3] = 0.0; }
    if (init_labels) {
        for (int n = gt; n < N; n += gnt) lab[n] = init_labels[(size_t)init * N_in + n];
    } else {
        Rng rng(seed * 0x100000001B3ull + 1469598103934665603ull * (unsigned long long)(init + 1));
        double* d2 = w.red + (size_t)init * (N_in > GT ? N_in : GT);
        int first = (int)(rng.uniform() * N); if (first >= N) first = N - 1;
        if (rank == 0) for (int d = threadIdx.x; d < D; d += GT) cent[d] = xs[(size_t)first * D + d];
        cl.sync();
        // k-means++: one D^2-weighted draw per further centre
        for (int c = 1; c < K; ++c) {
            for (int n = gw; n < N; n += gnw) {
                double sq = 0;
                for (int d = lane; d < D; d += 32) { const double t = xs[(size_t)n * D + d] - cent[(c - 1) * D + d]; sq = fma(t, t, sq); }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                if (lane == 0) d2[n] = (c == 1) ? sq : fmin(d2[n], sq);
            }
            cl.sync();
            const double u = rng.uniform();   // every CTA draws, so the generators stay in step
            if (rank == 0) {
                const int chunk = (N + GT - 1) / GT, beg = threadIdx.x * chunk, end = min(beg + chunk, N);
                double cs = 0;
                for (int n = beg; n < end; ++n) cs += d2[n];
                s_part[threadIdx.x] = cs;
                if (threadIdx.x == 0) s_pick = N - 1;
                __syncthreads();
                if (threadIdx.x == 0) {
                    double total = 0;
                    for (int t = 0; t < GT; ++t) total += s_part[t];
                    const double thr = u * total;
                    double run = 0; int t = 0;
                    for (; t < GT; ++t) { if (run + s_part[t] >= thr) break; run += s_part[t]; }
                    if (t < GT) {
                        int b2 = t * chunk, e2 = min(b2 + chunk, N), n = b2;
                        for (; n < e2; ++n) { run += d2[n]; if (run >= thr) break; }
                        s_pick = min(n, N - 1);
                    }
                }
                __syncthreads();
                for (int d = threadIdx.x; d < D; d += GT) cent[c * D + d] = xs[(size_t)s_pick * D + d];
            }
            cl.sync();
        }
        // Lloyd iterations (sklearn KMeans: max_iter 300, tol 1e-4 * mean feature variance; X is standardised)
        for (int n = gt; n < N; n += gnt) lab[n] = -1;
        cl.sync();
        int cur = 0;
        const int nr = 1 + (D + 31) / 32;       // rounds per cluster: the count, then 32 features at a time
        for (int it = 0; it < 300; ++it) {
            const double* cc = cent + (size_t)cur * K * D;
            double* cn = cent + (size_t)(cur ^ 1) * K * D;
            int changed = 0;
            for (int n = gw; n < N; n += gnw) {
                double best = DBL_MAX; int bk = 0;
                for (int k = 0; k < K; ++k) {
                    double sq = 0;
                    for (int d = lane; d < D; d += 32) { const double t = xs[(size_t)n * D + d] - cc[k * D + d]; sq = fma(t, t, sq); }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                    if (sq < best) { best = sq; bk = k; }
                }
                if (lane == 0 && lab[n] != bk) { lab[n] = bk; changed = 1; }
            }
            changed = __syncthreads_or(changed);
            if (threadIdx.x == 0) chg[rank] = changed;
            cl.sync();
            int any = 0;
            for (int i = 0; i < CLI; ++i) any |= chg[i];
            // counts and coordinate sums: (cluster k, round) pairs are dealt to the CTAs; inside a CTA warp w takes the samples
            // w, w + nw, ..., the lanes take the features, per-warp partials are added in warp order
            for (int p = rank; p < K * nr; p += CLI) {
                const int k = p / nr, round = p % nr;
                const int d = (round - 1) * 32 + lane;
                double a = 0;
                if (round == 0) { if (lane == 0) for (int n = wid; n < N; n += nw) a += lab[n] == k ? 1.0 : 0.0; }
                else if (d < D) for (int n = wid; n < N; n += nw) if (lab[n] == k) a += xs[(size_t)n * D + d];
                s_acc[wid][lane] = a;
                __syncthreads();
                if (wid == 0 && (round == 0 ? lane == 0 : d < D)) {
                    double t = 0;
                    for (int i = 0; i < nw; ++i) t += s_acc[i][lane];
                    tot[k * (1 + D) + (round == 0 ? 0 : 1 + d)] = t;
                }
                __syncthreads();
            }
            cl.sync();
            // shift (every CTA computes the same number) and the next centres (written by CTA 0 into the other buffer)
            double sh = 0;
            for (int i = threadIdx.x; i < K * D; i += GT) {
                const int k = i / D, d = i % D;
                const double cnt = tot[k * (1 + D)];
                double v = cc[i];
                if (cnt > 0) { v = tot[k * (1 + D) + 1 + d] / cnt; const double t = v - cc[i]; sh += t * t; }
                if (rank == 0) cn[i] = v;
            }
            sh = block_sum_d(sh, s_red);
            cur ^= 1;
            cl.sync();
            if (!any || sh <= 1e-4) break;
        }
    }
    cl.sync();
    double* sresp = w.sresp + (size_t)init * N_in * K;
    for (int i = gt; i < N * K; i += gnt) { const double r = (lab[i / K] == i % K) ? 1.0 : 0.0; resp[i] = r; sresp[i] = r; }
}

// nk and means of every (restart, component): grid (K, n_init, ceil(D / 32)), 1024 threads.  Warp w takes the samples w, w + 32,
// ...; its lanes 32 features; the 32 per-warp partials are added in warp order (the result does not depend on scheduling).
__global__ void __launch_bounds__(1024) k_big_means(int N_in, const int* n_dev, int D, int K, GmmWs w)
{
    const int k = blockIdx.x, init = blockIdx.y;
    if (w.state[init * 4 + 1] != 0.0) return;
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const double* resp = w.resp + (size_t)init * N_in * K;
    double* par = w.par + (size_t)init * pstride(K, D);
    double* wts = par; double* mu = par + K;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __shared__ double s_acc[32][33];
    __shared__ double s_nk;
    {
        double t = 0;
        for (int n = threadIdx.x; n < N; n += 1024) t += resp[(size_t)n * K + k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) s_acc[wid][0] = t;
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0;
            for (int i = 0; i < 32; ++i) a += s_acc[i][0];
            s_nk = a + 10 * DBL_EPSILON;
            if (blockIdx.z == 0) wts[k] = s_nk;   // nk; divided by N once the covariance has used it (k_big_chol)
        }
        __syncthreads();
    }
    const int d = blockIdx.z * 32 + lane;
    double a = 0;
    if (d < D)
        for (int n = wid; n < N; n += 32) a = fma(resp[(size_t)n * K + k], w.xs[(size_t)n * D + d], a);
    s_acc[wid][lane] = a;
    __syncthreads();
    if (wid == 0 && d < D) {
        double t = 0;
        for (int i = 0; i < 32; ++i) t += s_acc[i][lane];
        mu[k * D + d] = t / s_nk;
    }
}

// per (restart, component): covariance from the split-K Gram partials, Cholesky factor (to global memory for k_big_inv), log-determinant
// + log weight.  One CTA of 1024 threads; L lives in shared memory as a packed lower triangle (row i at i (i + 1) / 2).
__global__ void __launch_bounds__(1024) k_big_chol(int N_in, const int* n_dev, int D, int K, double reg, GmmWs w)
{
    extern __shared__ double Ls[];
    const int k = blockIdx.x, init = blockIdx.y;
    if (w.state[init * 4 + 1] != 0.0) return;
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    double* par = w.par + (size_t)init * pstride(K, D);
    double* wts = par;
    double* Cm = par + K + K * D + (size_t)k * D * D;                       // out: covariance
    const double* G = w.gram + ((size_t)init * K + k) * KS * D * D;
    const int T = blockDim.x, tid = threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5, nw = T >> 5;
    const double nk = wts[k];
    __shared__ int s_bad;
    __shared__ double s_ld[32];
    if (tid == 0) s_bad = 0;
    // covariance: the Gram partials are added in split order; only tiles on or above the diagonal were computed, so (a, b) with
    // a > b is read from (b, a)
    for (int i = tid; i < D * D; i += T) {
        const int a = i / D, b = i % D;
        const int src = a <= b ? a * D + b : b * D + a;
        double g = 0;
        for (int sp = 0; sp < KS; ++sp) g += G[(size_t)sp * D * D + src];
        const double c = g / nk + (a == b ? reg : 0.0);
        Cm[i] = c;
        if (b <= a) Ls[a * (a + 1) / 2 + b] = c;
    }
    __syncthreads();
    // blocked right-looking Cholesky on the packed lower triangle, panels of PB columns, three block-wide barriers per PANEL:
    //   (a) the PB x PB diagonal block, unblocked, by one warp (lane = row of the block, warp barriers only)
    //   (b) the panel below it: every row solves its own small triangular system against the finished diagonal block
    //   (c) the trailing matrix takes the rank-PB update, a warp per row with the row's panel entries in registers
    constexpr int PB = 16;
    auto idx = [](int i, int c) { return i * (i + 1) / 2 + c; };
    for (int j0 = 0; j0 < D; j0 += PB) {
        const int jb = min(PB, D - j0);
        if (wid == 0) {
            for (int jj = 0; jj < jb; ++jj) {
                const int j = j0 + jj;
                const double d = Ls[idx(j, j)];          // the same value in every lane
                if (!(d > 0)) { if (lane == 0) s_bad = 1; break; }
                const double piv = sqrt(d);
                __syncwarp();
                double lij = 0.0;
                const bool below = lane > jj && lane < jb;
                if (below) { lij = Ls[idx(j0 + lane, j)] / piv; Ls[idx(j0 + lane, j)] = lij; }
                if (lane == jj) Ls[idx(j, j)] = piv;
                __syncwarp();
                if (below)
                    for (int c = jj + 1; c <= lane; ++c) Ls[idx(j0 + lane, j0 + c)] = fma(-lij, Ls[idx(j0 + c, j)], Ls[idx(j0 + lane, j0 + c)]);
                __syncwarp();
            }
        }
        __syncthreads();
        if (s_bad) break;
        for (int i = j0 + jb + tid; i < D; i += T) {
            double x[PB];
            const int ri = idx(i, j0);
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (c < jb) {
                    double acc = Ls[ri + c];
                    const int rc = idx(j0 + c, j0);
#pragma unroll
                    for (int pp = 0; pp < PB; ++pp) if (pp < c) acc = fma(-x[pp], Ls[rc + pp], acc);
                    x[c] = acc / Ls[rc + c];
                }
            }
#pragma unroll
            for (int c = 0; c < PB; ++c) if (c < jb) Ls[ri + c] = x[c];
        }
        __syncthreads();
        for (int i = j0 + jb + wid; i < D; i += nw) {
            const int ri = idx(i, 0);
            double li[PB];
#pragma unroll
            for (int pp = 0; pp < PB; ++pp) li[pp] = pp < jb ? Ls[ri + j0 + pp] : 0.0;
            for (int c = j0 + jb + lane; c <= i; c += 32) {
                const int rc = idx(c, j0);
                double acc = Ls[ri + c];
#pragma unroll
                for (int pp = 0; pp < PB; ++pp) if (pp < jb) acc = fma(-li[pp], Ls[rc + pp], acc);
                Ls[ri + c] = acc;
            }
        }
        __syncthreads();
    }
    __syncthreads();
    if (s_bad) {
        if (tid == 0) { w.state[init * 4 + 1] = 1.0; w.state[init * 4 + 3] = 1.0; } // done, failed
        return;
    }
    // log|prec_chol| + log weight; the factor goes to global memory (the slot of this pair's first Gram partial, which is dead now) for
    // the inversion kernel, which spreads the independent columns of L^-1 over several CTAs
    double* Lg = w.gram + ((size_t)init * K + k) * KS * D * D;
    for (int i = tid; i < D * (D + 1) / 2; i += T) Lg[i] = Ls[i];
    if (wid == 0) {
        double ld = 0;
        for (int j = lane; j < D; j += 32) ld -= log(Ls[j * (j + 1) / 2 + j]);
        s_ld[lane] = ld;
        __syncwarp();
        if (lane == 0) {
            double t = 0;
            for (int i = 0; i < 32; ++i) t += s_ld[i];
            w.ldw[init * K + k] = t + log(nk / N);
        }
    }
    __syncthreads();   // every thread has read nk = wts[k]
    if (tid == 0) wts[k] = nk / N;
}

// prec_chol = (L^-1)^T of one (restart, component) pair, the columns of Z = L^-1 dealt round-robin to CHOL_SPLIT CTAs x 32 warps:
//     Z[c][c] = 1 / L[c][c],   Z[r][c] = -(sum_{p=c}^{r-1} L[r][p] Z[p][c]) / L[r][r]   (r > c)
// forward substitution, one warp per column c with the column in registers (lane l holds Z[c + l + 32 q][c]).  Column c of Z is row c of
// U (upper triangular); the warp writes the whole row, zeros below the diagonal included (the E-step multiplies by the whole matrix).
constexpr int CHOL_SPLIT = 4;
__global__ void __launch_bounds__(1024) k_big_inv(int D, int K, GmmWs w)
{
    extern __shared__ double Ls[];
    const int k = blockIdx.x, init = blockIdx.y, part = blockIdx.z;
    if (w.state[init * 4 + 1] != 0.0) return;
    double* par = w.par + (size_t)init * pstride(K, D);
    double* U = par + K + K * D + (size_t)K * D * D + (size_t)k * D * D;
    const double* Lg = w.gram + ((size_t)init * K + k) * KS * D * D;
    const int T = blockDim.x, tid = threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5, nw = T >> 5;
    __shared__ double s_col[DBIG];
    for (int i = tid; i < D * (D + 1) / 2; i += T) Ls[i] = Lg[i];
    __syncthreads();
    // reciprocals of the diagonal (the forward substitution multiplies instead of dividing 189 times per column)
    for (int j = tid; j < D; j += T) s_col[j] = 1.0 / Ls[j * (j + 1) / 2 + j];
    __syncthreads();
    constexpr int ZQ = (DBIG + 31) / 32;
    for (int c = wid * CHOL_SPLIT + part; c < D; c += nw * CHOL_SPLIT) {
        double z[ZQ];
#pragma unroll
        for (int q = 0; q < ZQ; ++q) z[q] = 0.0;
        if (lane == 0) z[0] = s_col[c];
        for (int r = c + 1; r < D; ++r) {
            const int rr = r * (r + 1) / 2;
            double sum = 0;
#pragma unroll
            for (int q = 0; q < ZQ; ++q) {
                const int pp = c + lane + 32 * q;
                if (pp < r) sum = fma(Ls[rr + pp], z[q], sum);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const double val = -sum * s_col[r];
            const int owner = (r - c) & 31, slot = (r - c) >> 5;
#pragma unroll
            for (int q = 0; q < ZQ; ++q) if (q == slot && lane == owner) z[q] = val;
        }
        for (int pp = lane; pp < c; pp += 32) U[(size_t)c * D + pp] = 0.0;
#pragma unroll
        for (int q = 0; q < ZQ; ++q) {
            const int pp = c + lane + 32 * q;
            if (pp < D) U[(size_t)c * D + pp] = z[q];
        }
    }
}

// b = mu U of every (restart, component): four lanes per column, each over a quarter of the rows
__global__ void __launch_bounds__(1024) k_big_bvec(int D, int K, GmmWs w)
{
    const int k = blockIdx.x, init = blockIdx.y;
    if (w.state[init * 4 + 1] != 0.0) return;
    const double* par = w.par + (size_t)init * pstride(K, D);
    const double* mu = par + K + (size_t)k * D;
    const double* U = par + K + K * D + (size_t)K * D * D + (size_t)k * D * D;
    for (int j4 = threadIdx.x; j4 < 4 * ((D + 7) / 8) * 8; j4 += blockDim.x) {
        const int j = j4 >> 2, part = j4 & 3;
        double a = 0;
        if (j < D)
            for (int i = part; i <= j; i += 4) a = fma(mu[i], U[(size_t)i * D + j], a);
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        if (j < D && part == 0) w.bvec[((size_t)init * K + k) * D + j] = a;
    }
}

// E-step after the GEMM: warp per sample; log N_k from |Y[r,k][n] - b[r,k]|^2, responsibilities, per-block log-likelihood sums
__global__ void __launch_bounds__(256) k_big_estep(int N_in, const int* n_dev, int D, int K, GmmWs w)
{
    const int init = blockIdx.y;
    if (w.state[init * 4 + 1] != 0.0) return;
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int n = blockIdx.x * 8 + wl;
    __shared__ double s_lse[8];
    double lse = 0.0;
    if (n < N) {
        double lw[KMAX];
        double mx = -DBL_MAX;
        for (int k = 0; k < K; ++k) {
            const double* y = w.big + (((size_t)init * K + k) * N_in + n) * D;
            const double* b = w.bvec + ((size_t)init * K + k) * D;
            double q = 0;
            for (int j = lane; j < D; j += 32) { const double t = y[j] - b[j]; q = fma(t, t, q); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            lw[k] = -0.5 * (D * 1.8378770664093453 + q) + w.ldw[init * K + k];
            mx = fmax(mx, lw[k]);
        }
        double s = 0;
        for (int k = 0; k < K; ++k) s += exp(lw[k] - mx);
        lse = mx + log(s);
        if (lane == 0)
            for (int k = 0; k < K; ++k) {
                const double r = exp(lw[k] - lse);
                w.resp[((size_t)init * N_in + n) * K + k] = r;
                w.sresp[((size_t)init * N_in + n) * K + k] = sqrt(r);
            }
    }
    if (lane == 0) s_lse[wl] = lse;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int i = 0; i < 8; ++i) t += s_lse[i];
        w.lowpart[(size_t)init * ((N_in + 7) / 8) + blockIdx.x] = t;
    }
}

// after E + M: the lower bound of this iteration, convergence, bookkeeping (sklearn: the M-step runs before the test)
__global__ void k_big_converge(int N_in, const int* n_dev, int D, int K, int n_init, int it, int max_iter, double tol, GmmWs w)
{
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int init = threadIdx.x;
    const int nblk = (N + 7) / 8, stride = (N_in + 7) / 8;
    __shared__ int s_running;
    if (threadIdx.x == 0) s_running = 0;
    __syncthreads();
    if (init < n_init) {
        double* st = w.state + init * 4;
        double* tail = w.par + (size_t)init * pstride(K, D) + K + K * D + 2 * (size_t)K * D * D;
        if (st[1] == 0.0) {
            double t = 0;
            for (int i = 0; i < nblk; ++i) t += w.lowpart[(size_t)init * stride + i];
            const double lower = t / N;
            const bool conv = it > 1 && fabs(lower - st[0]) < tol;
            st[0] = lower;
            tail[0] = lower; tail[1] = (double)it; tail[2] = conv ? 1.0 : 0.0; tail[3] = 1.0;
            if (conv || it >= max_iter) st[1] = 1.0; else atomicAdd(&s_running, 1);
        } else if (st[3] != 0.0) {
            tail[0] = -DBL_MAX; tail[3] = 0.0; // a covariance was not positive definite
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) *w.flag = s_running;
}

// the restart with the largest lower bound among those that did not fail (-1: all failed) -> w.flag[0]
__global__ void k_big_best(int D, int K, int n_init, GmmWs w)
{
    const int ps = pstride(K, D);
    int best = -1;
    double bl = 0;
    for (int i = 0; i < n_init; ++i) {
        const double* tail = w.par + (size_t)i * ps + K + K * D + 2 * (size_t)K * D * D;
        if (tail[3] != 0.0 && (best < 0 || tail[0] > bl)) { best = i; bl = tail[0]; }
    }
    *w.flag = best;
}

// what k_big_proba copies out after a fit: scaler, the winning restart's parameters and its index (out == nullptr: nothing)
struct ParamExport { const double* scale; const double* par; int best; double* out; };

// predict_proba from Y = X U ([K, N_in, D]: component k's rows at Y + k N_in D), b_k = mu_k U_k ([K, D]) and the per-component
// constants c ([K]: log|prec_chol_k| + log w_k, or whatever else does not depend on the sample); warp per sample
__global__ void __launch_bounds__(256) k_big_proba(int N_in, const int* n_dev, int D, int K, const double* __restrict__ Y,
                                                   const double* __restrict__ bvec, const double* __restrict__ cvec, double* proba,
                                                   ParamExport ex)
{
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int n = blockIdx.x * 8 + wl;
    if (n < N) {
        double lw[KMAX];
        double mx = -DBL_MAX;
        for (int k = 0; k < K; ++k) {
            const double* y = Y + ((size_t)k * N_in + n) * D;
            const double* b = bvec + (size_t)k * D;
            double q = 0;
            for (int j = lane; j < D; j += 32) { const double t = y[j] - b[j]; q = fma(t, t, q); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            lw[k] = -0.5 * (D * 1.8378770664093453 + q) + cvec[k];
            mx = fmax(mx, lw[k]);
        }
        double s = 0;
        for (int k = 0; k < K; ++k) s += exp(lw[k] - mx);
        const double lse = mx + log(s);
        if (lane == 0)
            for (int k = 0; k < K; ++k) proba[(size_t)n * K + k] = exp(lw[k] - lse);
    }
    if (blockIdx.x == 0 && ex.out) {
        const int ps = pstride(K, D);
        for (int i = threadIdx.x; i < 2 * D; i += blockDim.x) ex.out[i] = ex.scale[i];
        for (int i = threadIdx.x; i < ps; i += blockDim.x) ex.out[2 * D + i] = ex.par[i];
        if (threadIdx.x == 0) ex.out[2 * D + ps] = (double)ex.best;
    }
}

static int fit_big(int N, const int* n_dev, int D, int K, int n_init, int max_iter, double tol, double reg, unsigned long long seed,
                   const int* init_labels, GmmWs& w, cudaStream_t st, int* best_out)
{
    ISB_REQUIRE(n_init <= 1024, "too many restarts");
    const int RK = n_init * K;
    const size_t sND = (size_t)N * D, sDD = (size_t)D * D;
    const int ps = pstride(K, D);
    const size_t chol_smem = sizeof(double) * (size_t)D * (D + 1) / 2;
    ISB_CUDA_CHECK(cudaFuncSetAttribute(k_big_chol, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_smem));
    ISB_CUDA_CHECK(cudaFuncSetAttribute(k_big_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_smem));
    auto m_step = [&]() -> int {
        k_big_means<<<dim3(K, n_init, (D + 31) / 32), 1024, 0, st>>>(N, n_dev, D, K, w);
        ISB_LAUNCH_CHECK();
        // split-K partial Gram matrices (tiles on or above the diagonal); k_big_chol adds them
        {
            const BatchStride bs = { 0, 0, 0, 0, (size_t)K * KS * sDD, (size_t)KS * sDD, sDD };
            const FuseW fw = { w.sresp, w.par + K, (size_t)N * K, K, (size_t)ps, D };
            k_dgemm_batched<true, true><<<dim3((D + TN - 1) / TN, (D + TM - 1) / TM, RK * KS), 256, 0, st>>>(
                w.xs, D, w.xs, D, w.gram, D, bs, D, D, N, n_dev, 0, w.state, K, 1, KS, 0, fw);
            ISB_LAUNCH_CHECK();
        }
        k_big_chol<<<dim3(K, n_init), 1024, chol_smem, st>>>(N, n_dev, D, K, reg, w);
        ISB_LAUNCH_CHECK();
        k_big_inv<<<dim3(K, n_init, CHOL_SPLIT), 1024, chol_smem, st>>>(D, K, w);
        ISB_LAUNCH_CHECK();
        k_big_bvec<<<dim3(K, n_init), 1024, 0, st>>>(D, K, w);
        ISB_LAUNCH_CHECK();
        return ISB_OK;
    };
    k_big_init<<<n_init * CLI, GT, 0, st>>>(N, n_dev, D, K, seed, init_labels, w);
    ISB_LAUNCH_CHECK();
    if (int rc = m_step()) return rc;
    for (int it = 1; it <= max_iter; ++it) {
        {
            const BatchStride bs = { 0, 0, (size_t)ps, sDD, (size_t)K * sND, sND, 0 };
            k_dgemm_batched<false, false><<<dim3((D + TN - 1) / TN, (N + TM - 1) / TM, RK), 256, 0, st>>>(
                w.xs, D, w.par + K + K * D + (size_t)K * sDD, D, w.big, D, bs, N, D, D, n_dev, 1, w.state, K, 0, 1, 1, FuseW());
            ISB_LAUNCH_CHECK();
        }
        k_big_estep<<<dim3((N + 7) / 8, n_init), 256, 0, st>>>(N, n_dev, D, K, w);
        ISB_LAUNCH_CHECK();
        if (int rc = m_step()) return rc;
        k_big_converge<<<1, 1024, 0, st>>>(N, n_dev, D, K, n_init, it, max_iter, tol, w);
        ISB_LAUNCH_CHECK();
        int running = 0;
        ISB_CUDA_CHECK(cudaMemcpyAsync(&running, w.flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        ISB_CUDA_CHECK(cudaStreamSynchronize(st));
        if (running == 0) break;
    }
    k_big_best<<<1, 1, 0, st>>>(D, K, n_init, w);
    ISB_LAUNCH_CHECK();
    ISB_CUDA_CHECK(cudaMemcpyAsync(best_out, w.flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    ISB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (*best_out >= 0) {
        // Y = X U of the winner into the first K slots of the big buffer
        const BatchStride bs = { 0, 0, 0, sDD, 0, sND, 0 };
        k_dgemm_batched<false, false><<<dim3((D + TN - 1) / TN, (N + TM - 1) / TM, K), 256, 0, st>>>(
            w.xs, D, w.par + (size_t)*best_out * ps + K + K * D + (size_t)K * sDD, D, w.big, D, bs, N, D, D, n_dev, 1, nullptr, K, 0, 1, 1, FuseW());
        ISB_LAUNCH_CHECK();
    }
    return ISB_OK;
}

// select the best restart, evaluate predict_proba for every sample, export the parameters
__global__ void __launch_bounds__(256) k_gmm_predict(int N_in, const int* n_dev, int D, int K, int n_init, GmmWs w, double* proba,
                                                    double* params_out)
{
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const int ps = pstride(K, D);
    int best = -1;
    double bl = 0;
    for (int i = 0; i < n_init; ++i) {
        const double* tail = w.par + (size_t)i * ps + K + K * D + 2 * (size_t)K * D * D;
        if (tail[3] != 0.0 && (best < 0 || tail[0] > bl)) { best = i; bl = tail[0]; }
    }
    __shared__ double s_logdet[KMAX];
    if (best < 0) { // every restart hit a singular covariance: NaN probabilities make the failure visible
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * K; i += gridDim.x * blockDim.x) proba[i] = nan("");
        if (blockIdx.x == 0 && threadIdx.x == 0 && params_out) params_out[2 * D + ps - 1] = 0.0;
        return;
    }
    const double* par = w.par + (size_t)best * ps;
    const double* wts = par; const double* mu = par + K; const double* pc = mu + K * D + (size_t)K * D * D;
    if (threadIdx.x < K) {
        double ld = 0;
        for (int j = 0; j < D; ++j) ld += log(pc[(size_t)threadIdx.x * D * D + j * D + j]);
        s_logdet[threadIdx.x] = ld + log(wts[threadIdx.x]);
    }
    __syncthreads();
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
        double lw[KMAX];
        double lse = log_prob_all(w.xs + (size_t)n * D, D, K, wts, mu, pc, s_logdet, lw);
        for (int k = 0; k < K; ++k) proba[(size_t)n * K + k] = exp(lw[k] - lse);
    }
    if (blockIdx.x == 0 && params_out) {
        for (int i = threadIdx.x; i < 2 * D; i += blockDim.x) params_out[i] = w.scale[i];
        for (int i = threadIdx.x; i < ps; i += blockDim.x) params_out[2 * D + i] = par[i];
        if (threadIdx.x == 0) params_out[2 * D + ps] = (double)best;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// predict_proba of a GIVEN model (isb_gmm_predict): a fitted GaussianMixture / BayesianGaussianMixture of any covariance type,
// optionally behind a StandardScaler, packed on the host into one vector
//     shift[D] | scale[D] | U[K, D, D] (upper-triangular precision Cholesky factors, zeros below) | b[K, D] = mu_k U_k | c[K]
// lw_k = -1/2 (D log 2 pi + |x U_k - b_k|^2) + c_k with x = (nan -> 0 (f) - shift) / scale;  proba = softmax(lw).
// Rows at or beyond the (device) sample count are neither read nor written.
// ---------------------------------------------------------------------------------------------------------------------

__host__ __device__ inline int model_len(int D, int K) { return 2 * D + K * D * D + K * D + K; }

// D <= DMAX: one thread per sample, the model in shared memory, the standardised row and the K log-densities in registers
// (every loop runs to its compile-time bound under a guard, so nothing is indexed at run time)
constexpr int PT = 128;
__global__ void __launch_bounds__(PT) k_model_predict(const double* __restrict__ feat, int N_in, int D, int ld, const int* n_dev, int K,
                                                     const double* __restrict__ model, double* proba)
{
    __shared__ double s_m[2 * DMAX + KMAX * DMAX * DMAX + KMAX * DMAX + KMAX];
    const int len = model_len(D, K);
    for (int i = threadIdx.x; i < len; i += PT) s_m[i] = model[i];
    __syncthreads();
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const double* shift = s_m;
    const double* scale = s_m + D;
    const double* U = s_m + 2 * D;
    const double* b = U + K * D * D;
    const double* c = b + K * D;
    for (int n = blockIdx.x * PT + threadIdx.x; n < N; n += gridDim.x * PT) {
        double x[DMAX];
#pragma unroll
        for (int i = 0; i < DMAX; ++i) {
            double f = 0.0;
            if (i < D) {
                f = feat[(size_t)n * ld + i];
                f = isnan(f) ? 0.0 : f;
                f = (f - shift[i]) / scale[i];
            }
            x[i] = f;
        }
        double lw[KMAX];
        double mx = -DBL_MAX;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            lw[k] = -DBL_MAX;
            if (k < K) {
                const double* Uk = U + k * D * D;
                double q = 0;
#pragma unroll
                for (int j = 0; j < DMAX; ++j) {
                    if (j < D) {
                        double y = 0;
#pragma unroll
                        for (int i = 0; i <= j; ++i) y = fma(x[i], Uk[i * D + j], y);
                        y -= b[k * D + j];
                        q = fma(y, y, q);
                    }
                }
                lw[k] = -0.5 * (D * 1.8378770664093453 + q) + c[k];
                mx = fmax(mx, lw[k]);
            }
        }
        double s = 0;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) if (k < K) s += exp(lw[k] - mx);
        const double lse = mx + log(s);
#pragma unroll
        for (int k = 0; k < KMAX; ++k) if (k < K) proba[(size_t)n * K + k] = exp(lw[k] - lse);
    }
}

// DMAX < D: the standardised, NaN-cleaned rows [N, D] for the GEMM (rows below the sample count only)
__global__ void __launch_bounds__(256) k_model_standardise(const double* __restrict__ feat, int N_in, int D, int ld, const int* n_dev,
                                                           const double* __restrict__ model, double* __restrict__ xs)
{
    const int N = n_dev ? min(*n_dev, N_in) : N_in;
    const size_t total = (size_t)N * D;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int n = (int)(i / D), d = (int)(i % D);
        double f = feat[(size_t)n * ld + d];
        f = isnan(f) ? 0.0 : f;
        xs[i] = (f - model[d]) / model[D + d];
    }
}

static size_t carve_predict(void* ws, size_t bytes, int N, int D, int K, double** xs, double** ys)
{
    if (D <= DMAX) return 0;
    WsCarver c(ws, bytes);
    *xs = c.take<double>((size_t)N * D);
    *ys = c.take<double>((size_t)K * N * D);
    return isb_align(c.off);
}

static size_t carve_gmm(GmmWs& w, void* ws, size_t bytes, int N, int D, int K, int n_init)
{
    WsCarver c(ws, bytes);
    w.xs = c.take<double>((size_t)N * D);
    w.scale = c.take<double>(2 * (size_t)D);
    w.resp = c.take<double>((size_t)n_init * N * K);
    w.lab = c.take<int>((size_t)n_init * N);
    w.par = c.take<double>((size_t)n_init * pstride(K, D));
    w.red = c.take<double>((size_t)n_init * (N > GT ? N : GT));
    if (D > DMAX) {
        w.big = c.take<double>((size_t)n_init * K * N * D);
        w.bvec = c.take<double>((size_t)n_init * K * D);
        w.ldw = c.take<double>((size_t)n_init * K);
        w.lowpart = c.take<double>((size_t)n_init * ((N + 7) / 8));
        w.cent = c.take<double>((size_t)n_init * 2 * K * D);
        w.iflag = c.take<int>((size_t)n_init * CLI);
        w.gram = c.take<double>((size_t)n_init * K * KS * D * D);
        w.sresp = c.take<double>((size_t)n_init * N * K);
        w.tot = c.take<double>((size_t)n_init * K * (1 + D));
        w.state = c.take<double>((size_t)n_init * 4);
        w.flag = c.take<int>(1);
    }
    return isb_align(c.off);
}

} // namespace

extern "C" size_t isb_gmm_workspace_bytes(int N, int D, int K, int n_init)
{
    GmmWs w;
    return carve_gmm(w, nullptr, 0, N, D, K, n_init);
}

extern "C" int isb_gmm_params_len(int D, int K) { return 2 * D + pstride(K, D) + 1; }

extern "C" int isb_gmm_fit_predict(const double* feat, int N, int D, int ld, const int32_t* n_dev, int K, int n_init, int max_iter,
                                   double tol, double reg_covar, int use_scaler, unsigned long long seed, const int32_t* init_labels,
                                   double* proba, double* params_out, void* ws, size_t ws_bytes, isb_stream_t stream)
{
    ISB_REQUIRE(feat && proba && ws, "null pointer");
    ISB_REQUIRE(N > 0 && D > 0 && ld >= D && K > 0 && n_init > 0 && max_iter > 0, "bad sizes");
    if (D > DBIG || K > KMAX) { isb_set_error("device GMM handles D <= %d and K <= %d (got D=%d K=%d)", DBIG, KMAX, D, K); return ISB_ERR_UNSUPPORTED; }
    GmmWs w;
    size_t need = carve_gmm(w, ws, ws_bytes, N, D, K, n_init);
    ISB_REQUIRE(need <= ws_bytes, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(ISB_PROF_GMM, st);
    if (D > DMAX) {
        int best = -1;
        k_big_scale<<<(D + 31) / 32, 1024, 0, st>>>(feat, N, n_dev, D, ld, use_scaler, w);
        ISB_LAUNCH_CHECK();
        if (int rc = fit_big(N, n_dev, D, K, n_init, max_iter, tol, reg_covar, seed, init_labels, w, st, &best)) return rc;
        if (best >= 0) {
            const ParamExport ex = { w.scale, w.par + (size_t)best * pstride(K, D), best, params_out };
            k_big_proba<<<(N + 7) / 8, 256, 0, st>>>(N, n_dev, D, K, w.big, w.bvec + (size_t)best * K * D, w.ldw + (size_t)best * K, proba,
                                                     ex);
            ISB_LAUNCH_CHECK();
            return ISB_OK;
        }
        // every restart failed: fall through to k_gmm_predict, which reports it (NaN probabilities, ok = 0)
    } else {
        k_gmm_scale<<<D, GT, 0, st>>>(feat, N, n_dev, D, ld, use_scaler, w);
        ISB_LAUNCH_CHECK();
        // one thread-block cluster per restart; the cluster size follows the (upper bound of the) sample count
        const int CL = N <= 1024 ? 1 : (N <= 4096 ? 2 : (N <= 16384 ? 4 : 8));
        const size_t par_bytes = sizeof(double) * (size_t)pstride(K, D);
        ISB_CUDA_CHECK(cudaFuncSetAttribute(k_gmm_fit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)par_bytes));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(n_init * CL); cfg.blockDim = dim3(GT); cfg.dynamicSmemBytes = par_bytes; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        ISB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, k_gmm_fit, N, n_dev, D, K, max_iter, tol, reg_covar, seed, init_labels, CL, w));
        ISB_LAUNCH_CHECK();
    }
    int blocks = (N + 255) / 256;
    if (blocks > 148) blocks = 148;
    k_gmm_predict<<<blocks, 256, 0, st>>>(N, n_dev, D, K, n_init, w, proba, params_out);
    ISB_LAUNCH_CHECK();
    return ISB_OK;
}

extern "C" int isb_gmm_model_len(int D, int K) { return model_len(D, K); }

extern "C" size_t isb_gmm_predict_workspace_bytes(int N, int D, int K)
{
    double *xs, *ys;
    return carve_predict(nullptr, 0, N, D, K, &xs, &ys);
}

extern "C" int isb_gmm_predict(const double* feat, int N, int D, int ld, const int32_t* n_dev, int K, const double* model, double* proba,
                               void* ws, size_t ws_bytes, isb_stream_t stream)
{
    ISB_REQUIRE(feat && model && proba, "null pointer");
    ISB_REQUIRE(N > 0 && D > 0 && ld >= D && K > 0, "bad sizes");
    if (D > DBIG || K > KMAX) { isb_set_error("device GMM handles D <= %d and K <= %d (got D=%d K=%d)", DBIG, KMAX, D, K); return ISB_ERR_UNSUPPORTED; }
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(ISB_PROF_GMM, st);
    if (D <= DMAX) {
        int blocks = (N + PT - 1) / PT;
        if (blocks > 4 * 148) blocks = 4 * 148;
        k_model_predict<<<blocks, PT, 0, st>>>(feat, N, D, ld, n_dev, K, model, proba);
        ISB_LAUNCH_CHECK();
        return ISB_OK;
    }
    double *xs = nullptr, *ys = nullptr;
    ISB_REQUIRE(ws, "null pointer");
    const size_t need = carve_predict(ws, ws_bytes, N, D, K, &xs, &ys);
    ISB_REQUIRE(need <= ws_bytes, "workspace too small");
    int blocks = (int)(((size_t)N * D + 255) / 256);
    if (blocks > 8 * 148) blocks = 8 * 148;
    k_model_standardise<<<blocks, 256, 0, st>>>(feat, N, D, ld, n_dev, model, xs);
    ISB_LAUNCH_CHECK();
    // Y_k = X U_k for every component in one launch (U_k upper triangular: column tiles skip the rows below them)
    const size_t sND = (size_t)N * D, sDD = (size_t)D * D;
    const BatchStride bs = { 0, 0, 0, sDD, 0, sND, 0 };
    k_dgemm_batched<false, false><<<dim3((D + TN - 1) / TN, (N + TM - 1) / TM, K), 256, 0, st>>>(
        xs, D, model + 2 * D, D, ys, D, bs, N, D, D, n_dev, 1, nullptr, K, 0, 1, 1, FuseW());
    ISB_LAUNCH_CHECK();
    const double* bvec = model + 2 * D + (size_t)K * sDD;
    const ParamExport none = { nullptr, nullptr, 0, nullptr };
    k_big_proba<<<(N + 7) / 8, 256, 0, st>>>(N, n_dev, D, K, ys, bvec, bvec + (size_t)K * D, proba, none);
    ISB_LAUNCH_CHECK();
    return ISB_OK;
}
