// kmeans.cu -- OPT-IN replacement for the cv2.kmeans call of stage 02 (02_color_extract.py:39-50; SURVEY 8f rank 2).
//
// The reference estimates the K Lab centres with cv2.kmeans (kmeans++ seeding, <= 40 Lloyd iterations, eps 0.5, best of 3
// attempts) on a seeded 200 000-pixel subsample: 0.26-0.29 s on the host per image, hundreds of times the GPU time of everything
// that follows.  cv2.kmeans draws from OpenCV's global RNG, so no other implementation can return its centres bit for bit; this
// one keeps the structure (same sample -- the caller passes the reference's own indices --, kmeans++ with 3 trials per centre,
// Lloyd to the same stopping rule, best of `attempts` by compactness) and is DETERMINISTIC: the sample's 8-bit Lab values are
// accumulated as integers, the compactness in fixed point, so no result depends on the order of the atomics.
// Contract: the centres and the compactness are pinned bit for bit to oracle/kmeans_model.py, a NumPy restatement of these kernels
// (tests/test_gpu_kmeans_exact.py; exact because of --fmad=false, integer sums and the fixed-point compactness), and their
// compactness is within 2 % of cv2.kmeans' on the same sample (tests/test_gpu_kmeans.py); labels and masks then follow from the
// usual exact assignment to THESE centres.  Off by default: the drop-in stage script uses it only when OMNI_B200_KMEANS=gpu.
//
// Every (frame, attempt) pair is an independent RUN with its own state and seeding scratch; all runs of a chunk of frames go
// through the same launches (run index = blockIdx.y of the Lloyd assignment, one CTA per run in the seeding, one thread per run in
// the update), so a batch of frames costs about as many launches as one frame.  A run's arithmetic does not depend on the other
// runs or on the grid, so omni_kmeans_lab (one frame) and every frame of omni_kmeans_lab_batch give the same bits.
#include "fast_device.cuh"

#define KM_MAX_K OMNI_MAX_K
#define KM_THREADS 256
#define KM_SEED_THREADS 1024
#define KM_TRIALS 3                       // candidates per new centre in the seeding (OpenCV's generateCentersPP uses 3, too)
#define KM_FIX 1024.0f                    // compactness in 1 / 1024 units (u64)
#define KM_CHUNK_BYTES ((size_t)256 << 20) // workspace of one chunk of frames (include/omni_b200.h omni_kmeans_lab_batch)

struct KmState {                          // device block of one k-means run (one attempt on one frame)
    float ctr[KM_MAX_K * 3];              // current centres
    unsigned int sum[KM_MAX_K * 4];       // per centre: sum L, sum a, sum b, count (integers: order-independent)
    unsigned long long comp;              // compactness of the last assignment (fixed point)
    int converged;
};

struct KmBest {                           // result of one frame: the most compact of its attempts
    float ctr[KM_MAX_K * 3];
    unsigned long long comp;              // fixed point; ~0: none
};

__device__ __forceinline__ unsigned long long km_mix(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__device__ __forceinline__ double km_uniform(unsigned long long seed, unsigned a, unsigned b, unsigned c)
{
    const unsigned long long r = km_mix(seed ^ km_mix(((unsigned long long)a << 40) ^ ((unsigned long long)b << 20) ^ c));
    return (double)(r >> 11) * (1.0 / 9007199254740992.0);
}

// sample[f][i] = 8-bit Lab of pixel idx[i] of frame f = blockIdx.y (idx == NULL: pixel i), packed L | a << 8 | b << 16
__global__ void __launch_bounds__(KM_THREADS) fk_km_gather(const u8 *__restrict__ px, size_t frame_stride, int w, size_t pitch,
                                                           const int *__restrict__ idx, int n, const u16 *__restrict__ labtab,
                                                           u32 *__restrict__ sample)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = idx ? idx[i] : i;
    const int y = p / w, x = p - y * w;
    const u8 *q = px + (size_t)blockIdx.y * frame_stride + (size_t)y * pitch + 3 * (size_t)x;
    int L, a, b;
    lab_noclamp(labtab, labtab + 256, q[0], q[1], q[2], L, a, b);
    sample[(size_t)blockIdx.y * n + i] = (u32)L | ((u32)a << 8) | ((u32)b << 16);
}

__device__ __forceinline__ float km_d2(u32 s, float c0, float c1, float c2)
{
    const float d0 = (float)(s & 255u) - c0, d1 = (float)((s >> 8) & 255u) - c1, d2 = (float)((s >> 16) & 255u) - c2;
    return d0 * d0 + d1 * d1 + d2 * d2;
}

// kmeans++ seeding, one CTA per run (run r = frame r / attempts, attempt r % attempts): the first centre uniformly at random, every
// further one the best of KM_TRIALS candidates drawn with probability proportional to the squared distance to the nearest centre
// so far.  dist: n floats of scratch per run.
__global__ void __launch_bounds__(KM_SEED_THREADS) fk_km_seed(const u32 *__restrict__ samples, int n, int K, unsigned long long seed,
                                                               int attempts, float *__restrict__ dists, KmState *__restrict__ runs)
{
    __shared__ double s_thr[KM_SEED_THREADS];          // per-thread sums of dist[] (the coarse level of the cumulative distance)
    __shared__ double s_red[KM_SEED_THREADS];
    __shared__ int s_pick[KM_TRIALS];
    __shared__ double s_pot[KM_TRIALS];
    const int run = blockIdx.x, attempt = run % attempts;
    const u32 *sample = samples + (size_t)(run / attempts) * n;
    float *dist = dists + (size_t)run * n;
    KmState *S = runs + run;
    const int tid = threadIdx.x;
    const int per = (n + KM_SEED_THREADS - 1) / KM_SEED_THREADS, lo = min(n, tid * per), hi = min(n, lo + per);
    auto block_sum = [&](double v) {                   // fixed-shape tree: the same bits on every run
        s_red[tid] = v;
        __syncthreads();
        for (int d = KM_SEED_THREADS / 2; d > 0; d >>= 1) {
            if (tid < d) s_red[tid] += s_red[tid + d];
            __syncthreads();
        }
        const double t = s_red[0];
        __syncthreads();
        return t;
    };
    if (tid == 0) {
        const int first = min(n - 1, (int)(km_uniform(seed, attempt, 0, 0) * n));
        const u32 s = sample[first];
        S->ctr[0] = (float)(s & 255u); S->ctr[1] = (float)((s >> 8) & 255u); S->ctr[2] = (float)((s >> 16) & 255u);
    }
    __syncthreads();
    double mine = 0.0;
    {
        const float c0 = S->ctr[0], c1 = S->ctr[1], c2 = S->ctr[2];
        for (int i = lo; i < hi; i++) { const float d = km_d2(sample[i], c0, c1, c2); dist[i] = d; mine += d; }
    }
    s_thr[tid] = mine;
    double total = block_sum(mine);
    for (int k = 1; k < K; k++) {
        // ---- draw the candidates: position r in the cumulative distance (thread sums first, then inside that thread's range) ----
        if (tid < KM_TRIALS) {
            const double r = km_uniform(seed, attempt, k, tid + 1) * total;
            double acc = 0.0;
            int th = KM_SEED_THREADS - 1;
            for (int i = 0; i < KM_SEED_THREADS; i++) { if (acc + s_thr[i] > r) { th = i; break; } acc += s_thr[i]; }
            const int a = min(n, th * per), b = min(n, a + per);
            int pick = max(a, b - 1);
            for (int i = a; i < b; i++) { acc += dist[i]; if (acc > r) { pick = i; break; } }
            s_pick[tid] = min(max(pick, 0), n - 1);
        }
        __syncthreads();
        // ---- potential of each candidate ----
        for (int t = 0; t < KM_TRIALS; t++) {
            const u32 s = sample[s_pick[t]];
            const float c0 = (float)(s & 255u), c1 = (float)((s >> 8) & 255u), c2 = (float)((s >> 16) & 255u);
            double pot = 0.0;
            for (int i = lo; i < hi; i++) pot += fminf(dist[i], km_d2(sample[i], c0, c1, c2));
            const double p = block_sum(pot);
            if (tid == 0) s_pot[t] = p;
        }
        __syncthreads();
        int bt = 0;
        for (int t = 1; t < KM_TRIALS; t++) if (s_pot[t] < s_pot[bt]) bt = t;
        const u32 s = sample[s_pick[bt]];
        const float c0 = (float)(s & 255u), c1 = (float)((s >> 8) & 255u), c2 = (float)((s >> 16) & 255u);
        if (tid == 0) { S->ctr[3 * k] = c0; S->ctr[3 * k + 1] = c1; S->ctr[3 * k + 2] = c2; }
        mine = 0.0;
        for (int i = lo; i < hi; i++) { const float d = fminf(dist[i], km_d2(sample[i], c0, c1, c2)); dist[i] = d; mine += d; }
        __syncthreads();
        s_thr[tid] = mine;
        total = block_sum(mine);
    }
    if (tid == 0) {
        S->converged = 0;
        S->comp = 0ull;
        for (int i = 0; i < KM_MAX_K * 4; i++) S->sum[i] = 0u;
    }
}

// one Lloyd assignment of run blockIdx.y: nearest centre (first minimum) of every sample, integer sums per centre, fixed-point
// compactness.  force: also runs that have converged (the final pass that measures the compactness of the final centres).
__global__ void __launch_bounds__(KM_THREADS) fk_km_assign(const u32 *__restrict__ samples, int n, int K, int attempts,
                                                           KmState *__restrict__ runs, int force)
{
    __shared__ float s_c[KM_MAX_K * 3];
    __shared__ unsigned int s_sum[KM_MAX_K * 4];
    __shared__ unsigned long long s_comp;
    KmState *S = runs + blockIdx.y;
    if (!force && S->converged) return;                              // uniform: the run has stopped, later launches are no-ops
    const u32 *sample = samples + (size_t)(blockIdx.y / attempts) * n;
    for (int i = threadIdx.x; i < K * 3; i += blockDim.x) s_c[i] = S->ctr[i];
    for (int i = threadIdx.x; i < K * 4; i += blockDim.x) s_sum[i] = 0u;
    if (threadIdx.x == 0) s_comp = 0ull;
    __syncthreads();
    unsigned long long comp = 0ull;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 s = sample[i];
        float bd = 3.0e38f;
        int best = 0;
        for (int k = 0; k < K; k++) {
            const float d = km_d2(s, s_c[3 * k], s_c[3 * k + 1], s_c[3 * k + 2]);
            if (d < bd) { bd = d; best = k; }
        }
        atomicAdd(&s_sum[4 * best], s & 255u);
        atomicAdd(&s_sum[4 * best + 1], (s >> 8) & 255u);
        atomicAdd(&s_sum[4 * best + 2], (s >> 16) & 255u);
        atomicAdd(&s_sum[4 * best + 3], 1u);
        comp += (unsigned long long)(bd * KM_FIX + 0.5f);
    }
    atomicAdd(&s_comp, comp);
    __syncthreads();
    for (int i = threadIdx.x; i < K * 4; i += blockDim.x)
        if (s_sum[i]) atomicAdd(&S->sum[i], s_sum[i]);
    if (threadIdx.x == 0 && s_comp) atomicAdd(&S->comp, s_comp);
}

// one thread per run: centres <- means; stop when no centre moved by more than eps (cv2's rule) -- an empty cluster keeps its centre
__global__ void fk_km_update(int n_runs, int K, float eps2, KmState *__restrict__ runs)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    KmState *S = runs + r;
    if (S->converged) return;
    float shift = 0.f;
    for (int k = 0; k < K; k++) {
        const unsigned cnt = S->sum[4 * k + 3];
        if (cnt) {
            float d2 = 0.f;
            for (int d = 0; d < 3; d++) {
                const float c = (float)((double)S->sum[4 * k + d] / (double)cnt);
                const float dd = c - S->ctr[3 * k + d];
                d2 += dd * dd;
                S->ctr[3 * k + d] = c;
            }
            shift = fmaxf(shift, d2);
        }
    }
    for (int i = 0; i < KM_MAX_K * 4; i++) S->sum[i] = 0u;
    S->comp = 0ull;
    if (shift <= eps2) S->converged = 1;
}

// one thread per frame, after the final (forced) assignment of every run: the attempts in order, each kept if strictly more compact
// than the best so far (ties: the lowest attempt)
__global__ void fk_km_keep_best(int n_frames, int attempts, int K, const KmState *__restrict__ runs, KmBest *__restrict__ best)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    KmBest *B = best + f;
    unsigned long long bc = ~0ull;
    int ba = -1;
    for (int a = 0; a < attempts; a++)
        if (runs[(size_t)f * attempts + a].comp < bc) { bc = runs[(size_t)f * attempts + a].comp; ba = a; }
    B->comp = bc;
    for (int i = 0; i < K * 3; i++) B->ctr[i] = ba >= 0 ? runs[(size_t)f * attempts + ba].ctr[i] : __int_as_float(-1);
}

// Body of omni_kmeans_lab / omni_kmeans_lab_batch (capi.cu checks the arguments).  n_frames frames at d_bgr + f * frame_stride share
// the sample indices h_idx (host, n of them) or NULL (every pixel, n = h * w).  h_centers: [n_frames][K][3]; h_compactness:
// [n_frames] or NULL.  Frames go through in chunks whose workspace (slot 6) stays within KM_CHUNK_BYTES, or one frame if that needs more.
int kmeans_lab_batch(omni_ctx *ctx, const u8 *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch, const int *h_idx,
                     int n, int K, int attempts, int max_iter, float eps, unsigned long long seed, float *h_centers,
                     double *h_compactness, cudaStream_t st)
{
    (void)h;
    OMNI_CUDA(fast_tables());
    const u16 *labtab = fast_lab_table();
    if (!labtab) { omni_set_error("Lab tables not available"); return OMNI_ERR_CUDA; }
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    // slot 6 (edge run lists; idle outside the edge pass): [KmState runs | KmBest frames | idx n i32 | sample F n u32 | dist F A n f32]
    const size_t per_frame = attempts * (sizeof(KmState) + (size_t)n * 4) + sizeof(KmBest) + (size_t)n * 4;
    const size_t fixed = al((size_t)n * 4) + 4 * 256;
    int F = (int)std::min<size_t>((size_t)n_frames, std::max<size_t>(1, KM_CHUNK_BYTES > fixed ? (KM_CHUNK_BYTES - fixed) / per_frame : 1));
    F = std::min(F, 65535 / attempts);                                     // runs are blockIdx.y of the assignment
    const size_t o_best = al(sizeof(KmState) * (size_t)F * attempts), o_idx = o_best + al(sizeof(KmBest) * (size_t)F),
                 o_sample = o_idx + al((size_t)n * 4), o_dist = o_sample + al((size_t)F * n * 4),
                 total = o_dist + al((size_t)F * attempts * n * 4);
    int rc = omni_ws_reserve(ctx, 6, total);
    if (rc != OMNI_OK) return rc;
    u8 *base = (u8 *)ctx->ws[6];
    KmState *runs = (KmState *)base;
    KmBest *best = (KmBest *)(base + o_best);
    u32 *sample = (u32 *)(base + o_sample);
    float *dist = (float *)(base + o_dist);
    int *d_idx = nullptr;
    if (h_idx) {
        d_idx = (int *)(base + o_idx);
        OMNI_CUDA(cudaMemcpyAsync(d_idx, h_idx, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
    }
    std::vector<KmBest> hb((size_t)F);
    for (int f0 = 0; f0 < n_frames; f0 += F) {
        const int nf = std::min(F, n_frames - f0), nr = nf * attempts;
        {
            KScope ks(ctx, "kmeans_gather", st);
            fk_km_gather<<<dim3((n + KM_THREADS - 1) / KM_THREADS, nf), KM_THREADS, 0, st>>>(d_bgr + (size_t)f0 * frame_stride, frame_stride, w,
                                                                                             pitch, d_idx, n, labtab, sample);
            OMNI_CUDA(cudaGetLastError());
        }
        {
            KScope ks(ctx, "kmeans_seed", st);
            fk_km_seed<<<nr, KM_SEED_THREADS, 0, st>>>(sample, n, K, seed, attempts, dist, runs);
            OMNI_CUDA(cudaGetLastError());
        }
        // CTAs per run: about 8 per SM over all runs (any grid gives the same integer sums)
        const int bx = std::max(1, std::min((n + KM_THREADS - 1) / KM_THREADS, (persist_blocks(ctx, 8) + nr - 1) / nr));
        for (int it = 0; it < max_iter; it++) {
            KScope ks(ctx, "kmeans_lloyd", st);
            fk_km_assign<<<dim3(bx, nr), KM_THREADS, 0, st>>>(sample, n, K, attempts, runs, 0);
            fk_km_update<<<(nr + 127) / 128, 128, 0, st>>>(nr, K, eps * eps, runs);
            OMNI_CUDA(cudaGetLastError());
        }
        {
            KScope ks(ctx, "kmeans_lloyd", st);
            fk_km_assign<<<dim3(bx, nr), KM_THREADS, 0, st>>>(sample, n, K, attempts, runs, 1);     // compactness of the final centres
            fk_km_keep_best<<<(nf + 127) / 128, 128, 0, st>>>(nf, attempts, K, runs, best);
            OMNI_CUDA(cudaGetLastError());
        }
        OMNI_CUDA(cudaMemcpyAsync(hb.data(), best, sizeof(KmBest) * (size_t)nf, cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));              // the next chunk reuses the runs and the host copy
        for (int f = 0; f < nf; f++) {
            for (int i = 0; i < 3 * K; i++) h_centers[(size_t)(f0 + f) * 3 * K + i] = hb[f].ctr[i];
            if (h_compactness) h_compactness[f0 + f] = (double)hb[f].comp / (double)KM_FIX;
        }
    }
    return OMNI_OK;
}
