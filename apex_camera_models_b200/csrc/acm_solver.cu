// Fused linearisation kernel, deterministic reduction, device-resident Levenberg-Marquardt.
//
// ONE kernel (`lin_kernel`, launched cooperatively so that every block is resident) serves
//   * acm_linearize: one streaming pass over the resident correspondences -> <= 54 sums, and
//   * acm_lm_solve:  the WHOLE solve -- pass, reduction, cross-GPU sum, LM step, next pass ... --
//     without returning to the host (one launch, one read-back per solve).
//
// Per pass: every thread accumulates the normal equations of its grid-stride share in registers
// (cp.async ring), the block combines them (fixed shuffle tree + fixed warp order) and hands its
// partial to the *reducer* of each sum -- one pass: a warp of block j (sums wrap around when the grid is
// smaller); solve: the whole block j, its warps splitting the column of partials -- which adds the
// partials in a fixed order, exchanges the total with its twin on the other GPUs over NVLink peer
// memory (solve: stores it into every GPU's exchange buffer), and broadcasts the result to every block.
// All three hand-offs travel as "flag-in-data" cells (a double split over two 8-byte words, each
// carrying half of a 64-bit tag -- 8-byte accesses are single-copy atomic, so a reader that sees
// the tag sees the data): no fence, no atomic, no barrier, one L2 (or NVLink) trip per hand-off.
// Every block then takes the LM step redundantly out of its own shared memory -- same arithmetic,
// same inputs, hence identical decisions everywhere, on every block and on every GPU.
//
// Determinism: fixed grid, per-thread sequential accumulation, fixed combine order at every level,
// rank-ordered cross-GPU sum.  No floating-point atomics.  Results depend on the grid size only.
#include "acm_linearize.cuh"
#include "acm_reduce.cuh"
#include "acm_models.cuh"
#include "acm_pointjac.cuh"

#include <stdlib.h>

#include <chrono>
#include <vector>

struct LmState {
    double x[ACM_MAX_PARAMS], xt[ACM_MAX_PARAMS];
    double H[ACM_MAX_PARAMS * ACM_MAX_PARAMS], g[ACM_MAX_PARAMS];
    double lower[ACM_MAX_PARAMS], upper[ACM_MAX_PARAMS];
    double cost, lambda, nu;
    double pred, dnorm, xnorm;
    double cost_tol, param_tol, grad_tol;
    double initial_cost, n_valid;
    long long t_begin_ns, t_end_ns;  // %globaltimer at the first and after the last pass of a persistent solve
    int32_t max_iter, iterations, passes, status, done, first, P, pad;
};
static_assert(sizeof(LmState) <= 4096, "LmState must fit the context's 4 KiB slot");
static_assert(sizeof(LmState) % sizeof(double) == 0, "LmState is copied as doubles");

#define LM_STATUS_PEER_FAILURE 5

// ---------------------------------------------------------------------------------------
// LM step: serial algebra on P <= 9 unknowns out of shared memory.
// Divisions are hoisted into reciprocals (1/D_i, 1/L_ii): a serial f64 division costs ~250
// cycles and the first version spent most of its 12 us on ~50 of them.
// ---------------------------------------------------------------------------------------
struct LmWork {
    double Ht[ACM_MAX_PARAMS * ACM_MAX_PARAMS], A[ACM_MAX_PARAMS * ACM_MAX_PARAMS];
    double gt[ACM_MAX_PARAMS], invD[ACM_MAX_PARAMS], gs[ACM_MAX_PARAMS], st[ACM_MAX_PARAMS];
    double red[64];
};

// Cholesky solve of the damped, Jacobi-scaled system (P <= 9) by one thread: operands are pulled
// from the shared LmWork into registers once, the factorisation is fully unrolled (compile-time P),
// the result goes back to w->st.  Reciprocals of the diagonal replace the divisions of the
// substitutions (a dependent f64 division costs ~150 cycles).
template <int P>
__device__ __forceinline__ bool chol_solve_work(LmWork* w) {
    double L[P * (P + 1) / 2], inv[P], yv[P], x[P];
#pragma unroll
    for (int i = 0; i < P; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) L[i * (i + 1) / 2 + j] = w->A[i * P + j];
#pragma unroll
    for (int i = 0; i < P; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double sum = L[i * (i + 1) / 2 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) sum -= L[i * (i + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
            if (i == j) {
                if (!(sum > 0.0)) return false;
                // only 1 / L_ii is ever used.  The serial sqrt + division chain of the P pivots was a third of the step
                // (~300 cycles each); a MUFU-seeded rsqrt (<= 2 ulp, ~80 cycles) perturbs the step no more than the FMA
                // contraction of this file already does relative to the oracle's separately rounded operations.
                inv[i] = (sum > 1e-280 && sum < 1e280) ? acm_rsqrt(sum) : 1.0 / sqrt(sum);
            } else {
                L[i * (i + 1) / 2 + j] = sum * inv[j];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
        double sum = w->gs[i];
#pragma unroll
        for (int k = 0; k < i; ++k) sum -= L[i * (i + 1) / 2 + k] * yv[k];
        yv[i] = sum * inv[i];
    }
#pragma unroll
    for (int i = P - 1; i >= 0; --i) {
        double sum = yv[i];
#pragma unroll
        for (int k = i + 1; k < P; ++k) sum -= L[k * (k + 1) / 2 + i] * x[k];
        x[i] = sum * inv[i];
    }
#pragma unroll
    for (int i = 0; i < P; ++i) w->st[i] = x[i];
    return true;
}

__device__ inline double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Decision part of the step (thread 0): accept / reject the trial point, update the damping,
// test convergence.  Returns true when the trial point was accepted.  The gradient maximum is taken up front (P independent
// loads) so that it overlaps the division behind it: a dependent f64 operation costs ~20 cycles here.
template <int P>
__device__ __forceinline__ bool lm_decide(LmState* s, const LmWork* w, double cost_t) {
    double gmax = 0.0;
#pragma unroll
    for (int i = 0; i < P; ++i) gmax = fmax(gmax, fabs(w->gt[i]));
    s->passes++;
    if (!(cost_t == cost_t)) { s->status = 4; s->done = 1; return false; }  // NaN sums (NaN observations): stop
    if (s->first) {
        s->first = 0;
        s->initial_cost = cost_t;
        return true;
    }
    const bool small_step = s->dnorm <= s->param_tol * (s->xnorm + s->param_tol);
    if (s->pred > 0.0 && cost_t < s->cost) {
        const double rho = (s->cost - cost_t) / s->pred;
        const double dcost = s->cost - cost_t, cost_old = s->cost;
        const double q = 2.0 * rho - 1.0, f = 1.0 - q * q * q;
        s->lambda *= (f > 1.0 / 3.0) ? f : 1.0 / 3.0;
        s->nu = 2.0;
        if (s->lambda < 1e-15) s->lambda = 1e-15;
        if (dcost <= s->cost_tol * cost_old) { s->status = 0; s->done = 1; }
        else if (small_step) { s->status = 1; s->done = 1; }
        else if (gmax <= s->grad_tol) { s->status = 2; s->done = 1; }
        return true;
    }
    if (small_step) { s->status = 1; s->done = 1; }
    else {
        s->lambda *= s->nu; s->nu *= 2.0;
        if (s->lambda > 1e30) { s->status = 4; s->done = 1; }
    }
    return false;
}

// 1 / sqrt of a diagonal entry of H (Jacobi scaling); degenerate entries scale by 1
// (the fast value is computed unconditionally -- garbage outside its range, replaced behind a rarely taken branch -- so that
// two calls interleave instead of queueing behind each other's branches)
__device__ __forceinline__ double lm_inv_sqrt_diag(double h) {
    double r = acm_rsqrt(h);
    if (!(h > 1e-280 && h < 1e280)) {
        const double d = sqrt(h);
        r = (d > 1e-300) ? 1.0 / d : 1.0;
    }
    return r;
}

// Cooperative step on a state that already sits in shared memory (`sh`), with the reduced sums of
// the pass in w->red (the pass ran at the trial point sh->xt).  The arithmetic of every scalar is
// the same as in the serial reference (oracle/acm_oracle_solver.c), including the order of the few
// sums, so both walk the same trajectory.  Every thread of the block must call it (barriers
// inside); on return the state is consistent and visible to the whole block.
//
// Four barriers on the common path (round 1 took ten, and 5.4 k of the ~15 k fixed cycles of a pass):
//   thread 0     unpack (upper triangle only; w->Ht's other entries stay zero from the kernel start), decide, count the iteration
//   -- barrier --
//   P*P threads  accepted state <- trial state (mirroring the triangle), scaled damped matrix straight from the source
//                (every thread takes the rsqrt of the two diagonal entries it needs itself)
//   -- barrier --
//   thread 0     Cholesky solve (retry loop with a larger lambda: rare)
//   -- barrier --
//   warp 0       trial point, quadratic model, norms: lane i owns parameter i, values move by shuffle
//   -- barrier --
template <int M, int KIND>
__device__ __forceinline__ void lm_step_smem(LmState* sh, LmWork* w, int tid, long long* stamps = nullptr) {
    constexpr int P = LinOps<M, KIND>::P;
    __shared__ int flag_accept, flag_go;
    __shared__ double s_cost_t, s_cnt;
    if (sh->done) return;  // uniform: shared state, read after the caller's barrier
    if (tid == 0) {
        double cost_t, cnt;
        if (stamps) stamps[0] = clock64();
        LinOps<M, KIND>::template unpack<false>(w->red, sh->xt, w->Ht, w->gt, &cost_t, &cnt);
        s_cost_t = cost_t; s_cnt = cnt;
        if (stamps) stamps[1] = clock64();
        flag_accept = lm_decide<P>(sh, w, cost_t) ? 1 : 0;
        if (stamps) stamps[2] = clock64();
        int go = 0;   // 1: solve for the next trial point, -1 / 0: the solve is over
        if (!sh->done) {
            if (sh->iterations >= sh->max_iter) { sh->status = 3; sh->done = 1; go = -1; }
            else { sh->iterations++; go = 1; }
        }
        flag_go = go;
    }
    __syncthreads();
    const int accept = flag_accept;
    int go = flag_go;   // thread 0 rewrites the flag only behind the next barrier
    {
        // the source of (H, g) at the accepted point: the trial sums when the trial point was accepted, else the kept state
        const double* const Hs = accept ? w->Ht : sh->H;
        if (tid < P * P) {
            const int i = tid / P, j = tid - i * P;
            const double h = Hs[accept ? (i <= j ? tid : j * P + i) : tid];
            double dj = 0.0;
            if (go > 0) {
                // thread 0 (which factors next) takes one rsqrt, the others two independent ones
                dj = lm_inv_sqrt_diag(Hs[j * P + j]);
                const double di = (i == j) ? dj : lm_inv_sqrt_diag(Hs[i * P + i]);
                double a = h * di * dj;
                if (i == j) a += sh->lambda;
                w->A[tid] = a;
            }
            if (accept) sh->H[tid] = h;   // nobody reads sh->H in this phase when accept is set
            if (tid < P) {   // row 0: j == tid, so dj is this parameter's scale
                const double g = accept ? w->gt[tid] : sh->g[tid];
                if (go > 0) { w->invD[tid] = dj; w->gs[tid] = -g * dj; }
                if (accept) { sh->x[tid] = sh->xt[tid]; sh->g[tid] = g; }
            }
        }
        if (accept && tid == 0) { sh->cost = s_cost_t; sh->n_valid = s_cnt; }
    }
    __syncthreads();
    if (stamps && tid == 0) stamps[3] = clock64();
    if (go > 0) {
        for (;;) {
            if (tid == 0) {
                int r = 1;
                if (!chol_solve_work<P>(w)) {
                    sh->lambda *= sh->nu; sh->nu *= 2.0;
                    r = 0;
                    if (sh->lambda > 1e30) { sh->status = 4; sh->done = 1; r = -1; }
                    else if (sh->iterations >= sh->max_iter) { sh->status = 3; sh->done = 1; r = -1; }
                    else sh->iterations++;
                }
                flag_go = r;
                if (stamps) stamps[4] = clock64();
            }
            __syncthreads();
            go = flag_go;
            if (go != 0) break;
            // retry with the larger damping (rare: rank-deficient normal equations)
            if (tid < P * P) {
                const int i = tid / P, j = tid - i * P;
                double a = sh->H[tid] * w->invD[i] * w->invD[j];
                if (i == j) a += sh->lambda;
                w->A[tid] = a;
            }
            __syncthreads();   // also: everybody has read the flag before thread 0 writes it again
        }
        if (go > 0 && tid < 32) {
            double x_i = 0.0, dx_i = 0.0, g_i = 0.0;
            if (tid < P) {
                x_i = sh->x[tid]; g_i = sh->g[tid];
                const double xt = clampd(x_i + w->st[tid] * w->invD[tid], sh->lower[tid], sh->upper[tid]);
                sh->xt[tid] = xt;
                dx_i = xt - x_i;
            }
            double hd = 0.0;
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double dx_j = __shfl_sync(0xffffffffu, dx_i, j);
                if (tid < P) hd += sh->H[tid * P + j] * dx_j;
            }
            const double yv_i = dx_i * (g_i + 0.5 * hd);   // row of the quadratic model
            double xnorm = 0.0, dnorm = 0.0, pred = 0.0;
#pragma unroll
            for (int i = 0; i < P; ++i) {
                const double xs = __shfl_sync(0xffffffffu, x_i, i), ds = __shfl_sync(0xffffffffu, dx_i, i), ys = __shfl_sync(0xffffffffu, yv_i, i);
                xnorm += xs * xs; dnorm += ds * ds; pred -= ys;
            }
            if (tid == 0) { sh->xnorm = sqrt(xnorm); sh->pred = pred; }
            if (tid == 1) sh->dnorm = sqrt(dnorm);
        }
    }
    __syncthreads();
    if (stamps && tid == 0) stamps[5] = clock64();
}

// Stand-alone step kernel: used when an NCCL all-reduce sits between the pass and the step (ranks
// without NVLink peer buffers).
template <int M, int KIND>
__global__ void __launch_bounds__(128) lm_step_kernel(LmState* __restrict__ s, const double* __restrict__ red) {
    __shared__ LmState sh;
    __shared__ LmWork work;
    constexpr int NW = sizeof(LmState) / sizeof(double);
    double* shw = reinterpret_cast<double*>(&sh);
    const double* gw = reinterpret_cast<const double*>(s);
    for (int i = threadIdx.x; i < NW; i += blockDim.x) shw[i] = __ldcg(gw + i);
    for (int i = threadIdx.x; i < LinOps<M, KIND>::NACC; i += blockDim.x) work.red[i] = __ldcg(red + i);
    for (int i = threadIdx.x; i < ACM_MAX_PARAMS * ACM_MAX_PARAMS; i += blockDim.x) work.Ht[i] = 0.0;   // the step fills the non-zero upper triangle only
    __syncthreads();
    if (sh.done) return;
    lm_step_smem<M, KIND>(&sh, &work, threadIdx.x);
    double* gout = reinterpret_cast<double*>(s);
    for (int i = threadIdx.x; i < NW; i += blockDim.x) gout[i] = shw[i];
}

// ---------------------------------------------------------------------------------------
// Flag-in-data cells.  A double travels as two 8-byte words {data_lo32 | tag_lo32 << 32},
// {data_hi32 | tag_hi32 << 32}; a reader accepts the cell once both halves carry the expected
// 64-bit tag.  Tags are never reused (64-bit counters starting at 1; buffers start zeroed).
// The accesses are volatile = relaxed at system scope: they bypass L1 and are coherent across
// NVLink peers.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void ll_store(LLCell* p, double v, unsigned long long tag) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    const unsigned long long w0 = (b & 0xffffffffULL) | (tag << 32);
    const unsigned long long w1 = (b >> 32) | (tag & 0xffffffff00000000ULL);
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(w0), "l"(w1) : "memory");
}
__device__ __forceinline__ ulonglong2 ll_load(const LLCell* p) {
    ulonglong2 r;
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p) : "memory");
    return r;
}
__device__ __forceinline__ bool ll_ready(const ulonglong2 c, unsigned long long tag) {
    return ((c.x >> 32) == (tag & 0xffffffffULL)) && ((c.y >> 32) == (tag >> 32));
}
__device__ __forceinline__ double ll_value(const ulonglong2 c) {
    return __longlong_as_double((long long)((c.x & 0xffffffffULL) | (c.y << 32)));
}
__device__ __forceinline__ double acm_qnan() { return __longlong_as_double(0x7ff8000000000000LL); }

__device__ __forceinline__ unsigned long long acm_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

#define ACM_SPIN_LIMIT_CYCLES 4000000000LL  // ~2 s: a lost peer (or a bug) ends the solve instead of hanging the GPU

// Warp-collective: total of col[0..nb) -- lane-strided sequential sums, then the fixed shuffle tree --
// where the cells are filled by the other blocks of this grid.  BATCH cells per lane are polled per
// trip (8: one L2 round trip per 256 blocks; 16 pushed the Double Sphere solve kernel over its 170-register cap and
// the spill landed in the streaming loop).  The summation order does not depend on BATCH.
template <int BATCH>
__device__ __forceinline__ double warp_sum_cells(const LLCell* __restrict__ col, int nb, int lane, unsigned long long tag, bool& bad) {
    double a = 0.0;
    for (int b0 = lane; b0 < nb; b0 += 32 * BATCH) {
        ulonglong2 c[BATCH];
        unsigned pending = 0;
#pragma unroll
        for (int j = 0; j < BATCH; ++j) if (b0 + 32 * j < nb) pending |= 1u << j;
        const long long t0 = clock64();
        while (pending) {
#pragma unroll
            for (int j = 0; j < BATCH; ++j) if (pending & (1u << j)) c[j] = ll_load(col + b0 + 32 * j);
#pragma unroll
            for (int j = 0; j < BATCH; ++j) if ((pending & (1u << j)) && ll_ready(c[j], tag)) pending &= ~(1u << j);
            if (pending && clock64() - t0 > ACM_SPIN_LIMIT_CYCLES) { bad = true; break; }
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) if (b0 + 32 * j < nb) a += ll_value(c[j]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
    bad = __any_sync(0xffffffffu, bad);
    return __shfl_sync(0xffffffffu, a, 0);
}

// ---------------------------------------------------------------------------------------
// All-reduce over NVLink peer memory, one sum per warp.  Lane r < n_ranks stores this rank's
// value into cell [set][my rank][slot] of rank r's exchange buffer (a plain store to a peer-mapped
// address travels over NVLink) and polls cell [set][r][slot] of its own buffer; the values are then
// added in rank order, so the totals are bit-identical on every rank, which keeps the ranks' LM
// decisions in lock step.  Two cell sets alternate (seq & 1): a rank can run at most one exchange
// ahead of the slowest one, so it never overwrites a cell that is still being read.
// A time-out (or a peer's abort flag) raises the sticky abort flag in EVERY rank's buffer: all ranks
// leave with an error instead of drifting apart; the host must re-attach the peers afterwards.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ LLCell* peer_cell(unsigned char* buf, int set, int src_rank, int slot) {
    return reinterpret_cast<LLCell*>(buf + ACM_PEER_HEADER_BYTES) + ((size_t)(set * ACM_MAX_PEERS + src_rank) * ACM_PEER_SLOT_CELLS + slot);
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ double warp_peer_exchange(const PeerArgs& peer, unsigned long long seq, int slot, double v, int lane, bool& bad) {
    const int set = (int)(seq & 1ULL);
    double mine = 0.0;
    bool fail = false;
    if (lane < peer.n_ranks) {
        ll_store(peer_cell(peer.bufs[lane], set, peer.rank, slot), v, seq);
        const LLCell* src = peer_cell(peer.bufs[peer.rank], set, lane, slot);
        const unsigned long long* abort_word = reinterpret_cast<const unsigned long long*>(peer.bufs[peer.rank]);
        const long long t0 = clock64();
        unsigned polls = 0;
        for (;;) {
            const ulonglong2 c = ll_load(src);
            if (ll_ready(c, seq)) { mine = ll_value(c); break; }
            if ((++polls & 255u) == 0 && (ld_volatile_u64(abort_word) != 0ULL || clock64() - t0 > ACM_SPIN_LIMIT_CYCLES)) { fail = true; break; }
        }
    }
    fail = __any_sync(0xffffffffu, fail);
    if (fail) {
        if (lane < peer.n_ranks) st_volatile_u64(reinterpret_cast<unsigned long long*>(peer.bufs[lane]), 1ULL);  // sticky, every rank sees it
        bad = true;
        return acm_qnan();
    }
    double tot = 0.0;
    for (int r = 0; r < peer.n_ranks; ++r) tot += __shfl_sync(0xffffffffu, mine, r);
    return tot;
}

// ---------------------------------------------------------------------------------------
// Streaming part: per-model configuration
// ---------------------------------------------------------------------------------------
// Measured on 100 M points (scripts/lin_bench.py; GB/s register prefetch -> cp.async ring):
// DEPTH > 0 = every thread keeps that many packets in flight in a shared-memory ring fed by cp.async;
// 0 = the next packet is prefetched into registers.
//   DS 5.88 -> 6.24 TB/s (3 deep), EUCM 5.63 -> 5.79, UCM 5.83 -> 6.47 (2 deep), FOV 4.50 -> 4.97
//   (3 deep, 128 threads), RadTan 4.09 -> 4.25 (2 deep; 5.1 with the structured accumulation; 128-thread blocks capped at 168
//   registers for 12 warps/SM measured 4.2-4.8); Pinhole (already at 7.1 TB/s) is faster without the ring.
// PTS = points evaluated per loop trip and thread (2 = one 16-byte packet per array, 4 = two packets: four independent
// evaluation chains for the scheduler to interleave; needs an even DEPTH >= 2).
template <int M> struct LinStream { static constexpr int DEPTH = 0, BLOCK = 256, PTS = 2; };
template <> struct LinStream<ACM_MODEL_DOUBLE_SPHERE> { static constexpr int DEPTH = 3, BLOCK = 256, PTS = 2; };
template <> struct LinStream<ACM_MODEL_EUCM> { static constexpr int DEPTH = 3, BLOCK = 256, PTS = 2; };
template <> struct LinStream<ACM_MODEL_UCM> { static constexpr int DEPTH = 2, BLOCK = 256, PTS = 2; };
template <> struct LinStream<ACM_MODEL_FOV> { static constexpr int DEPTH = 4, BLOCK = 256, PTS = 4; };
template <> struct LinStream<ACM_MODEL_RADTAN> { static constexpr int DEPTH = 3, BLOCK = 256, PTS = 2; };
// KB (37 accumulators, 166 registers): 3 blocks of 128 threads.  Same-box A/B (scripts/ab_lin.sh; boxes of the pool differ by
// up to 40 % on this FP64-bound kernel, so only same-box comparisons count): register prefetch 4.42 TB/s, ring 1 deep 3.95,
// 2 deep 4.51, 3 deep 4.59; capped at 128 registers (4 blocks per SM, 36-byte spill) 4.19.
// Round 2, same-box A/B (profiles/r02_ab_pts4.log): four points per trip, FOV 5262 -> 5463 GB/s (2 deep), KB 4789 -> 4861 (4 deep);
// RadTan loses (5348 -> 5139 / 4255) and keeps two.  FOV in 256-thread blocks (the compiler then takes 126 registers instead of
// 96, two blocks per SM): 5365 -> 5667 GB/s 4 deep, 5535 2 deep (profiles/r02_ab_fov_occ*.log); capping the registers for more
// warps loses (80 registers, 24 warps: 5144); KB in 256-thread blocks is unchanged (4761 -> 4781).  RadTan (198 registers, one
// 256-thread block per SM, long_scoreboard 0.56 per issue with the ring 2 deep): 3 deep 5345 -> 5560, 4 deep 5561; two 128-thread
// blocks 4876 (profiles/r02_ab_radtan_ring.log).  Double Sphere (the headline kernel) does not move: 3 deep x 2 points 5931-5939, 4 deep x 4
// points 5941, 4 deep x 2 points 5926-5952 GB/s over 200 launches (profiles/r02_ab_ds_headline.log).
template <> struct LinStream<ACM_MODEL_KANNALA_BRANDT> { static constexpr int DEPTH = 4, BLOCK = 128, PTS = 4; };

// The solve form of the kernel (128-thread blocks) has its own ring depth / points per trip / register cap: it carries the trial
// parameters in registers (the one-pass form reads them from the constant bank) and peaks at 152-168 registers outside the
// streaming loop.  Default: three blocks per SM (<= 170 registers, no spill); the wide models (KB, RadTan) are left uncapped.
// Same-box A/B of two uncapped blocks per SM against three capped ones (profiles/r02_ab_lm_stream*.log, us per pass at
// 1.25 M / 10 M correspondences): Double Sphere 15.1 -> 13.9 / 67.7 -> 66.4 (taken); EUCM 13.7 -> 12.7 / 63.4 -> 64.3 and UCM
// 11.4 -> 10.4 / 62.2 -> 70.3 (better from L2, worse from HBM: kept at three); FOV worse at both.  Four points per trip fit
// 166 registers for Double Sphere but gain nothing (15.2 / 70.0).
template <int M> struct SolveStream {
    // Ring depth / points per trip of the solve, measured on their own (us per pass at 10 M correspondences,
    // profiles/r02_ab_lm_fov.log, r02_ab_lm_kb_rt.log): FOV with four points per trip spilled under the 170-register cap (20
    // bytes): two points, 3 deep = 95.7 -> 80.0; KB two points 3 deep (238 registers) 102.8 -> 98.6; RadTan 3 deep 94.0 -> 90.9
    // (capping either at 170 registers spills: RadTan 154.6).
    static constexpr bool WIDE_MODEL = (M == ACM_MODEL_FOV || M == ACM_MODEL_KANNALA_BRANDT || M == ACM_MODEL_RADTAN);
    static constexpr int DEPTH = WIDE_MODEL ? 3 : LinStream<M>::DEPTH;
    static constexpr int PTS = WIDE_MODEL ? 2 : LinStream<M>::PTS;
    static constexpr int MIN_BLOCKS = (M == ACM_MODEL_KANNALA_BRANDT || M == ACM_MODEL_RADTAN) ? 0 : (M == ACM_MODEL_DOUBLE_SPHERE ? 2 : 3);
    // from this many correspondences per GPU on, the solve runs one uncapped 256-thread block per SM instead (half the blocks to
    // reduce over, same warps): Double Sphere 68.3 -> 66.0 us per pass at 10 M, 37.8 -> 37.2 at 5 M, 22.1 -> 22.3 at 2.5 M, slower at 450; UCM and FOV lose
    // 10-15 % at 10 M, EUCM gains 0.5 % (profiles/r02_ab_lm_stream2.log, _stream3.log).  0 = never.
    static constexpr size_t WIDE_BLOCK_FROM = (M == ACM_MODEL_DOUBLE_SPHERE) ? 4000000 : 0;
};
template <int M, bool SOLVE> struct StreamCfg { static constexpr int DEPTH = LinStream<M>::DEPTH, PTS = LinStream<M>::PTS; };
template <int M> struct StreamCfg<M, true> { static constexpr int DEPTH = SolveStream<M>::DEPTH, PTS = SolveStream<M>::PTS; };

struct LinKernelArgs {
    LinParams hp;                 // parameters of a single evaluation (mode 0)
    LmState* lm;                  // device-resident LM state (modes 1, 2)
    int mode;                     // 0: one pass at hp -> out; 1: one pass at lm->xt (skipped when lm->done) -> out; 2: the whole LM solve
    int max_passes;               // mode 2
    PeerArgs peer;                // NVLink exchange (bufs == nullptr: single GPU, or the caller all-reduces `out` itself)
    const double2 *X, *Y, *Z, *U, *V;
    size_t n;
    double pen2x2;                // 2 * invalid_penalty^2: cost of one invalid point
    LLCell* partials;             // [NACC][gridDim.x] block partials
    LLCell* bcast;                // [64] totals, reducer blocks -> every block (mode 2, single GPU)
    unsigned long long tag0;      // first hand-off tag of this launch (mode 2 uses tag0 + pass)
    double* out;                  // [NACC] totals (modes 0, 1)
    long long* trace;             // debug (ACM_LM_TRACE=1): clock64 stamps of block 0, 6 per pass
    int trace_pass;               // debug (ACM_LM_TRACE=2): >= 0 = every block stamps %globaltimer at the start, after the stream and at the end of this pass
};

// One streaming pass of this block over its grid-stride share + the block partial (fixed shuffle tree, then the
// warps in order) handed to the reducers as tagged cells.
// PRIMED: the first DEPTH packets of this pass are already in flight (issued while the previous pass's sums travelled).
template <int M, int KIND, int BS, bool SOLVE>
__device__ __forceinline__ void lin_stream_pass(const LinKernelArgs& a, const LinParams& p_in, unsigned long long tag, bool primed, bool prime_next) {
    using LM_ = LinOps<M, KIND>;
    constexpr int NACC = LM_::NACC;
    constexpr int NWARP = BS / 32;
    constexpr int DEPTH = StreamCfg<M, SOLVE>::DEPTH;
    __shared__ double wsum[NWARP][NACC];
    extern __shared__ double2 lin_ring[];
    LinParams p = p_in;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = (int)gridDim.x;
    const size_t npairs = a.n >> 1;
    const size_t stride = (size_t)nb * BS;
    const size_t i0 = (size_t)blockIdx.x * BS + tid;

    // cp.async ring: every thread keeps DEPTH packets (5 x 16 B each) in flight in its own
    // shared-memory slots -- deeper than a register prefetch could afford -- and reads them back with
    // five conflict-free LDS.128.  Only the owning thread touches a slot, so wait_group is all the
    // synchronisation needed.  ring[stage][array][thread].
    const double2* const src[5] = {a.X, a.Y, a.Z, a.U, a.V};
    auto issue = [&](int stage, size_t idx) {
        if (idx < npairs) {
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&lin_ring[(stage * 5 + q) * BS + tid]);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src[q] + idx) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto prime = [&]() {
        if constexpr (DEPTH > 0) {
#pragma unroll
            for (int s = 0; s < DEPTH; ++s) issue(s, i0 + (size_t)s * stride);
        }
    };
    if (!primed) prime();

    double acc[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc[i] = 0.0;
    int cnt = 0;   // valid points, for the specialisations that count them in an int (LinIntCount)
    size_t i = i0;
    if constexpr (DEPTH > 0 && StreamCfg<M, SOLVE>::PTS == 4) {
        // two packets (four points) per trip: the four evaluation chains are independent, the points still enter every
        // accumulator in the same order as in the two-point form, so the sums are bit-identical
        static_assert(DEPTH % 2 == 0, "PTS = 4 consumes the ring two stages at a time");
        int stage = 0;
        auto ld = [&](int st, int q) { return lin_ring[(st * 5 + q) * BS + tid]; };
#pragma unroll 1
        while (i + stride < npairs) {
            asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH > 1 ? DEPTH - 2 : 0) : "memory");
            const double2 x0 = ld(stage, 0), y0 = ld(stage, 1), z0 = ld(stage, 2), u0 = ld(stage, 3), v0 = ld(stage, 4);
            const double2 x1 = ld(stage + 1, 0), y1 = ld(stage + 1, 1), z1 = ld(stage + 1, 2), u1 = ld(stage + 1, 3), v1 = ld(stage + 1, 4);
            lin_point<LM_>(acc, cnt, p, x0.x, y0.x, z0.x, u0.x, v0.x);
            lin_point<LM_>(acc, cnt, p, x0.y, y0.y, z0.y, u0.y, v0.y);
            lin_point<LM_>(acc, cnt, p, x1.x, y1.x, z1.x, u1.x, v1.x);
            lin_point<LM_>(acc, cnt, p, x1.y, y1.y, z1.y, u1.y, v1.y);
            issue(stage, i + (size_t)DEPTH * stride);
            issue(stage + 1, i + (size_t)(DEPTH + 1) * stride);
            stage = (stage + 2 == DEPTH) ? 0 : stage + 2;
            i += 2 * stride;
        }
        if (i < npairs) {   // odd number of packets: the last one alone
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            const double2 x0 = ld(stage, 0), y0 = ld(stage, 1), z0 = ld(stage, 2), u0 = ld(stage, 3), v0 = ld(stage, 4);
            lin_point<LM_>(acc, cnt, p, x0.x, y0.x, z0.x, u0.x, v0.x);
            lin_point<LM_>(acc, cnt, p, x0.y, y0.y, z0.y, u0.y, v0.y);
            i += stride;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if constexpr (DEPTH > 0) {
        int stage = 0;
#pragma unroll 1
        while (i < npairs) {
            asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH > 0 ? DEPTH - 1 : 0) : "memory");
            const double2 x = lin_ring[(stage * 5 + 0) * BS + tid], y = lin_ring[(stage * 5 + 1) * BS + tid],
                          z = lin_ring[(stage * 5 + 2) * BS + tid], u = lin_ring[(stage * 5 + 3) * BS + tid],
                          v = lin_ring[(stage * 5 + 4) * BS + tid];
            lin_point<LM_>(acc, cnt, p, x.x, y.x, z.x, u.x, v.x);
            lin_point<LM_>(acc, cnt, p, x.y, y.y, z.y, u.y, v.y);
            issue(stage, i + (size_t)DEPTH * stride);  // after the packet has been consumed
            stage = (stage + 1 == DEPTH) ? 0 : stage + 1;
            i += stride;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
        // Software-pipelined stream: the five 16-byte loads of the next pair of points are in flight
        // while the current pair is evaluated.
        double2 x, y, z, u, v;
        if (i < npairs) { x = __ldcs(a.X + i); y = __ldcs(a.Y + i); z = __ldcs(a.Z + i); u = __ldcs(a.U + i); v = __ldcs(a.V + i); }
#pragma unroll 1
        while (i < npairs) {
            const size_t nx = i + stride;
            const size_t j = nx < npairs ? nx : i;  // clamp: the tail re-reads its own (cached) packet
            const double2 x2 = __ldcs(a.X + j), y2 = __ldcs(a.Y + j), z2 = __ldcs(a.Z + j), u2 = __ldcs(a.U + j), v2 = __ldcs(a.V + j);
            lin_point<LM_>(acc, cnt, p, x.x, y.x, z.x, u.x, v.x);
            lin_point<LM_>(acc, cnt, p, x.y, y.y, z.y, u.y, v.y);
            x = x2; y = y2; z = z2; u = u2; v = v2;
            i = nx;
        }
    }
    unsigned long long npts = (i0 < npairs) ? 2ULL * (unsigned long long)((npairs - i0 + stride - 1) / stride) : 0ULL;
    if ((a.n & 1) && blockIdx.x == 0 && tid == 0) {
        const size_t t = a.n - 1;
        const double* Xs = reinterpret_cast<const double*>(a.X); const double* Ys = reinterpret_cast<const double*>(a.Y);
        const double* Zs = reinterpret_cast<const double*>(a.Z); const double* Us = reinterpret_cast<const double*>(a.U);
        const double* Vs = reinterpret_cast<const double*>(a.V);
        lin_point<LM_>(acc, cnt, p, Xs[t], Ys[t], Zs[t], Us[t], Vs[t]);
        npts += 1;
    }
    if constexpr (LinIntCount<LM_>::value) acc[LM_::COUNT] = (double)cnt;
    // invalid points carry the residual (pen, pen): cost += pen^2 per invalid point
    if (a.pen2x2 != 0.0) acc[LM_::COST] += a.pen2x2 * ((double)npts - acc[LM_::COUNT]);

    if (a.trace != nullptr && prime_next && blockIdx.x == 0 && tid == 0) a.trace[6 * (int)(tag - a.tag0) + 1] = clock64();
    // ---- block partial: warp totals, then the warps in order.
    // Warp totals: the shuffle tree costs 15 instructions per accumulator and warp (435 for Double Sphere: 1.2 us of every
    // pass with 12 warps per SM, measured with ACM_LM_TRACE).  Where the drained cp.async ring is large enough, the warp
    // transposes instead: lane L stores accumulator k at [k][(L + k) & 31] (conflict-free), lane k then adds row k with four
    // interleaved partial sums in a fixed order -- ~3 instructions per accumulator.  Deterministic either way.
    constexpr size_t kRingBytes = (size_t)DEPTH * 5 * BS * sizeof(double2);
    constexpr bool kTranspose = kRingBytes >= (size_t)NWARP * NACC * 32 * sizeof(double) && NACC <= 32;
    if constexpr (kTranspose) {
        __syncthreads();   // every warp has drained its ring slots: the ring is scratch now
        double* tr = reinterpret_cast<double*>(lin_ring) + (size_t)warp * NACC * 32;
#pragma unroll
        for (int k = 0; k < NACC; ++k) tr[k * 32 + ((lane + k) & 31)] = acc[k];
        __syncwarp();
        if (lane < NACC) {
            const double* row = tr + lane * 32;
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {   // element j of the row = the value of lane j, stored at column (j + lane) & 31
                s0 += row[(j + 0 + lane) & 31]; s1 += row[(j + 1 + lane) & 31];
                s2 += row[(j + 2 + lane) & 31]; s3 += row[(j + 3 + lane) & 31];
            }
            wsum[warp][lane] = (s0 + s1) + (s2 + s3);
        }
    } else {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
            double v = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) wsum[warp][k] = v;
        }
    }
    __syncthreads();
    if (tid < NACC) {
        double v = wsum[0][tid];
#pragma unroll
        for (int k = 1; k < NWARP; ++k) v += wsum[k][tid];
        ll_store(a.partials + (size_t)tid * nb + blockIdx.x, v, tag);
    }
    // the first packets of the next pass do not depend on its parameters: fetch them while the sums travel
    if (prime_next) prime();
    __syncthreads();  // wsum may be rewritten by the next pass
}

// One pass of the solve on this block: stream, reduce, (exchange,) collect the totals, LM step.
// Everything below the kernel is force-inlined on purpose: a real (ABI) call inside the pass loop stacks the callee's
// register frame on top of the caller's (measured with ptxas -v: +38 registers for a thin loop around a non-inlined pass
// body, +70 for non-inlined reducers under an inlined streaming loop), which costs the streaming loop a resident block.
// Returns false when the solve is over (uniform over the block -- and over the grid: every block holds the same state).
template <int M, int KIND, int BS, bool SOLVE>
__device__ __forceinline__ bool lin_pass(const LinKernelArgs& a, LmState* sh, LmWork* work, int pass) {
    using LM_ = LinOps<M, KIND>;
    constexpr int ND = LM_::ND;
    constexpr int NACC = LM_::NACC;
    constexpr int NWARP = BS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = (int)gridDim.x;
    const unsigned long long tag = a.tag0 + (unsigned long long)pass, seq = a.peer.seq + (unsigned long long)pass;

    LinParams p = a.hp;
    if (SOLVE) {
        if (sh->done || pass >= a.max_passes) return false;
        p.fx = sh->xt[0]; p.fy = sh->xt[1]; p.cx = sh->xt[2]; p.cy = sh->xt[3];
#pragma unroll
        for (int k = 0; k < ND; ++k) p.d[k] = sh->xt[4 + k];
        lin_derive(M, p);
    } else if (a.mode != 0) {
        // one round trip: the done flag and the trial parameters are fetched together
        const int done = a.lm->done;
        p.fx = a.lm->xt[0]; p.fy = a.lm->xt[1]; p.cx = a.lm->xt[2]; p.cy = a.lm->xt[3];
#pragma unroll
        for (int k = 0; k < ND; ++k) p.d[k] = a.lm->xt[4 + k];
        if (done) return false;  // converged earlier in this enqueue batch (uniform over the grid)
        lin_derive(M, p);
    }
    const bool tr = SOLVE && a.trace != nullptr && blockIdx.x == 0 && tid == 0;
    if (tr) a.trace[6 * pass + 0] = clock64();
    const bool trb = SOLVE && a.trace != nullptr && pass == a.trace_pass && tid == 0;
    if (trb) a.trace[12 * a.max_passes + 3 * (int)blockIdx.x + 0] = (long long)acm_globaltimer();
    lin_stream_pass<M, KIND, BS, SOLVE>(a, p, tag, SOLVE && pass > 0, SOLVE);
    if (tr) a.trace[6 * pass + 2] = clock64();
    if (trb) a.trace[12 * a.max_passes + 3 * (int)blockIdx.x + 1] = (long long)acm_globaltimer();

    const bool solve_peers = SOLVE && a.peer.bufs != nullptr;
    bool bad = false;
    if (SOLVE) {
        // ---- reducer blocks (solve): sum j belongs to block j % nb, whose warps split the nb cells between them so that
        // every lane polls at most 4 cells in ONE trip (444 blocks: two dependent L2 round trips with a single warp per sum);
        // the warp totals are added in warp order.  The host keeps nb >= NACC for the solve, so the loop runs once.
        __shared__ double wsum[NWARP];
        const int chunk = (nb + NWARP - 1) / NWARP;
#pragma unroll 1
        for (int slot = (int)blockIdx.x; slot < NACC; slot += nb) {
            const int c0 = warp * chunk, len = max(0, min(chunk, nb - c0));
            const double part = warp_sum_cells<4>(a.partials + (size_t)slot * nb + c0, len, lane, tag, bad);
            if (lane == 0) wsum[warp] = part;
            bad = __syncthreads_or(bad) != 0;
            if (warp == 0) {
                double tot = wsum[0];
#pragma unroll
                for (int k = 1; k < NWARP; ++k) tot += wsum[k];
                if (bad) tot = acm_qnan();
                if (solve_peers) {
                    // multi-GPU solve: the rank's total goes straight into every rank's exchange buffer; the blocks of every GPU
                    // collect from there (one hop less than exchanging here and re-broadcasting)
                    if (lane < a.peer.n_ranks) ll_store(peer_cell(a.peer.bufs[lane], (int)(seq & 1ULL), a.peer.rank, slot), tot, seq);
                } else if (lane == 0) {
                    ll_store(a.bcast + slot, tot, tag);
                }
            }
            if (slot + nb < NACC) __syncthreads();   // wsum is reused (block-uniform condition)
        }
    } else {
        // ---- reducer warps (one pass): sum j belongs to warp (j / nb) % NWARP of block j % nb
#pragma unroll 1
        for (int slot = (int)blockIdx.x + nb * warp; slot < NACC; slot += nb * NWARP) {
            double tot = warp_sum_cells<8>(a.partials + (size_t)slot * nb, nb, lane, tag, bad);
            if (bad) tot = acm_qnan();
            if (a.peer.bufs && !bad) tot = warp_peer_exchange(a.peer, seq, slot, tot, lane, bad);
            if (lane == 0) a.out[slot] = tot;
        }
    }
    if (!SOLVE) return false;
    if (tr) a.trace[6 * pass + 3] = clock64();

    // ---- every block: collect the totals, take the LM step out of shared memory
    int nan_seen = 0;
    if (solve_peers) {
        // n_ranks x NACC cells of this GPU's exchange buffer, spread over the threads of the block (<= 4 each, polled
        // together), staged in shared memory, then added in rank order: bit-identical on every block of every GPU
        constexpr int CELLS = (NACC * ACM_MAX_PEERS + BS - 1) / BS;
        __shared__ double xch[ACM_MAX_PEERS][NACC];
        const int set = (int)(seq & 1ULL);
        unsigned char* const mine = a.peer.bufs[a.peer.rank];
        const unsigned long long* abort_word = reinterpret_cast<const unsigned long long*>(mine);
        const int total = NACC * a.peer.n_ranks;
        ulonglong2 c[CELLS];
        unsigned pending = 0, polls = 0;
#pragma unroll
        for (int q = 0; q < CELLS; ++q) if (tid + q * BS < total) pending |= 1u << q;
        const long long t0 = clock64();
        while (pending) {
#pragma unroll
            for (int q = 0; q < CELLS; ++q)
                if (pending & (1u << q)) { const int i = tid + q * BS; c[q] = ll_load(peer_cell(mine, set, i / NACC, i % NACC)); }
#pragma unroll
            for (int q = 0; q < CELLS; ++q) if ((pending & (1u << q)) && ll_ready(c[q], seq)) pending &= ~(1u << q);
            if (pending && (++polls & 255u) == 0 && (ld_volatile_u64(abort_word) != 0ULL || clock64() - t0 > ACM_SPIN_LIMIT_CYCLES)) break;
        }
#pragma unroll
        for (int q = 0; q < CELLS; ++q) { const int i = tid + q * BS; if (i < total) xch[i / NACC][i % NACC] = ll_value(c[q]); }
        if (pending) {   // a peer is gone: raise the sticky abort flag on every rank
            for (int r = 0; r < a.peer.n_ranks; ++r) st_volatile_u64(reinterpret_cast<unsigned long long*>(a.peer.bufs[r]), 1ULL);
        }
        const int lost = __syncthreads_or(pending != 0u);
        if (tid < NACC) {
            double v = 0.0;
            for (int r = 0; r < a.peer.n_ranks; ++r) v += xch[r][tid];
            if (lost) v = acm_qnan();
            work->red[tid] = v; nan_seen = !(v == v);
        }
    } else if (tid < NACC) {
        const long long t0 = clock64();
        for (;;) {
            const ulonglong2 c = ll_load(a.bcast + tid);
            if (ll_ready(c, tag)) { const double v = ll_value(c); work->red[tid] = v; nan_seen = !(v == v); break; }
            if (clock64() - t0 > ACM_SPIN_LIMIT_CYCLES) { nan_seen = 1; break; }
        }
    }
    nan_seen = __syncthreads_or(nan_seen);
    if (tr) a.trace[6 * pass + 4] = clock64();
    if (nan_seen) {
        // a hand-off timed out or a sum is NaN: stop here (every block takes the same decision)
        if (tid == 0) { sh->passes++; sh->status = 4; sh->done = 1; }
        __syncthreads();
    } else {
        lm_step_smem<M, KIND>(sh, work, tid, (a.trace != nullptr && blockIdx.x == 0) ? a.trace + 6 * a.max_passes + 6 * pass : nullptr);
    }
    if (tr) a.trace[6 * pass + 5] = clock64();
    if (trb) a.trace[12 * a.max_passes + 3 * (int)blockIdx.x + 2] = (long long)acm_globaltimer();
    return true;
}

template <int M, int KIND, int BS, bool SOLVE>
__global__ void __launch_bounds__(BS, (SOLVE && BS == 128) ? SolveStream<M>::MIN_BLOCKS : 0) lin_kernel(const __grid_constant__ LinKernelArgs a) {
    static_assert(LinOps<M, KIND>::NACC <= 64, "hand-off layout assumes <= 64 accumulators");
    constexpr int NSTATE = sizeof(LmState) / sizeof(double);
    __shared__ LmState sh;
    __shared__ LmWork work;
    const int tid = threadIdx.x;
    if (!SOLVE) {
        lin_pass<M, KIND, BS, false>(a, &sh, &work, 0);
        return;
    }
    double* shw = reinterpret_cast<double*>(&sh);
    const double* gw = reinterpret_cast<const double*>(a.lm);
    for (int i = tid; i < NSTATE; i += BS) shw[i] = __ldcg(gw + i);
    for (int i = tid; i < ACM_MAX_PARAMS * ACM_MAX_PARAMS; i += BS) work.Ht[i] = 0.0;   // the step fills the non-zero upper triangle only
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) sh.t_begin_ns = (long long)acm_globaltimer();
#pragma unroll 1
    for (int pass = 0; lin_pass<M, KIND, BS, SOLVE>(a, &sh, &work, pass); ++pass) {}
    if constexpr (StreamCfg<M, SOLVE>::DEPTH > 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
    if (blockIdx.x == 0) {
        __syncthreads();
        if (tid == 0) {
            sh.t_end_ns = (long long)acm_globaltimer();
            if (a.peer.bufs && ld_volatile_u64(reinterpret_cast<const unsigned long long*>(a.peer.bufs[a.peer.rank])) != 0ULL) sh.status = LM_STATUS_PEER_FAILURE;
        }
        __syncthreads();
        double* gout = reinterpret_cast<double*>(a.lm);
        for (int i = tid; i < NSTATE; i += BS) gout[i] = shw[i];
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// Hand-off buffers of the kernel: [64 sums][blocks] partial cells + 64 broadcast cells, zeroed once
// (tags start at 1 and never repeat).
static int32_t ensure_ll(acm_ctx* ctx, size_t blocks) {
    const size_t cells = 64 * blocks + 64;
    if (ctx->lm_ll_cap >= cells) return ACM_OK;
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->d_lm_ll); ctx->d_lm_ll = nullptr; ctx->lm_ll_cap = 0;
    void* p = nullptr;
    int32_t rc = acm_device_malloc(ctx, &p, cells * sizeof(LLCell));
    if (rc) return rc;
    ACM_CUDA(ctx, cudaMemsetAsync(p, 0, cells * sizeof(LLCell), ctx->stream));
    ctx->d_lm_ll = static_cast<LLCell*>(p); ctx->lm_ll_cap = cells;
    return ACM_OK;
}

template <int M, int KIND, int BS, bool SOLVE>
static int32_t launch_lin_bs(acm_ctx* ctx, LinKernelArgs& a, const acm_points* xyz, const acm_points* uv) {
    const size_t ring_bytes = (size_t)StreamCfg<M, SOLVE>::DEPTH * 5 * BS * sizeof(double2);
    const void* fn = reinterpret_cast<const void*>(&lin_kernel<M, KIND, BS, SOLVE>);
    int bps = 0;
    int32_t rc = acm_kernel_blocks_per_sm(ctx, fn, BS, ring_bytes, &bps);
    if (rc) return rc;
    const size_t n = xyz->n;
    int grid = grid_for(ctx, (n >> 1) + 1, BS, bps);
    // the solve gives every sum its own reducer block (a few hundred correspondences would otherwise queue all sums on the
    // warps of one or two blocks: 6.4 k of the 15 k cycles of a pass at n = 450); blocks without points contribute zeros
    if (SOLVE && grid < LinOps<M, KIND>::NACC) grid = LinOps<M, KIND>::NACC;
    rc = ensure_ll(ctx, (size_t)ctx->sm_count * 16);
    if (rc) return rc;
    ACM_REQUIRE(ctx, (size_t)grid <= (size_t)ctx->sm_count * 16, "linearize: grid larger than the hand-off buffer");
    a.X = comp<double2>(xyz, 0); a.Y = comp<double2>(xyz, 1); a.Z = comp<double2>(xyz, 2);
    a.U = comp<double2>(uv, 0); a.V = comp<double2>(uv, 1);
    a.n = n;
    a.partials = ctx->d_lm_ll;
    a.bcast = ctx->d_lm_ll + (ctx->lm_ll_cap - 64);
    a.out = ctx->d_reduce;
    // tags: one per pass, never reused
    a.tag0 = ctx->lm_tag + 1;
    ctx->lm_tag += (SOLVE ? (unsigned long long)a.max_passes : 1ULL) + 1ULL;
    void* args[] = {&a};
    if (ctx->coop_launch) {
        ACM_CUDA(ctx, cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(BS), args, ring_bytes, ctx->stream));
        ctx->launches++;
    } else {
        // no cooperative launch on this device / configuration: the grid never exceeds the resident capacity computed above
        lin_kernel<M, KIND, BS, SOLVE><<<grid, BS, ring_bytes, ctx->stream>>>(a);
        ACM_CHECK_LAUNCH(ctx);
    }
    return ACM_OK;
}

// Block size per model: the accumulators of the wide models (KB: 37 doubles) push the
// kernel past 128 registers/thread; 128-thread blocks then pack one more block per SM.
// The solve runs 128-thread blocks, or 256 from SolveStream<M>::WIDE_BLOCK_FROM correspondences on.
template <int M, int KIND>
static int32_t launch_lin(acm_ctx* ctx, LinKernelArgs& a, const acm_points* xyz, const acm_points* uv) {
    if (a.mode != 2) return launch_lin_bs<M, KIND, LinStream<M>::BLOCK, false>(ctx, a, xyz, uv);
    if constexpr (SolveStream<M>::WIDE_BLOCK_FROM != 0) {
        if (xyz->n >= SolveStream<M>::WIDE_BLOCK_FROM) return launch_lin_bs<M, KIND, 256, true>(ctx, a, xyz, uv);
    }
    return launch_lin_bs<M, KIND, 128, true>(ctx, a, xyz, uv);
}

#define ACM_DISPATCH_LIN(model, kind, ...)                                                                       \
    do {                                                                                                         \
        if ((kind) == ACM_RESIDUAL_ALGEBRAIC) {                                                                  \
            constexpr int KIND = ACM_RESIDUAL_ALGEBRAIC;                                                         \
            switch (model) {                                                                                     \
                case ACM_MODEL_UCM: { constexpr int M = ACM_MODEL_UCM; __VA_ARGS__; break; }                     \
                case ACM_MODEL_EUCM: { constexpr int M = ACM_MODEL_EUCM; __VA_ARGS__; break; }                   \
                case ACM_MODEL_DOUBLE_SPHERE: { constexpr int M = ACM_MODEL_DOUBLE_SPHERE; __VA_ARGS__; break; } \
                default: return acm_fail(ctx, ACM_ERR_INVALID_ARG, "the algebraic residual exists only for UCM, EUCM and Double Sphere"); \
            }                                                                                                    \
        } else if ((kind) == ACM_RESIDUAL_PIXEL) {                                                               \
            constexpr int KIND = ACM_RESIDUAL_PIXEL;                                                             \
            switch (model) {                                                                                     \
                case ACM_MODEL_PINHOLE: { constexpr int M = ACM_MODEL_PINHOLE; __VA_ARGS__; break; }             \
                case ACM_MODEL_RADTAN: { constexpr int M = ACM_MODEL_RADTAN; __VA_ARGS__; break; }               \
                case ACM_MODEL_KANNALA_BRANDT: { constexpr int M = ACM_MODEL_KANNALA_BRANDT; __VA_ARGS__; break; } \
                case ACM_MODEL_UCM: { constexpr int M = ACM_MODEL_UCM; __VA_ARGS__; break; }                     \
                case ACM_MODEL_EUCM: { constexpr int M = ACM_MODEL_EUCM; __VA_ARGS__; break; }                   \
                case ACM_MODEL_DOUBLE_SPHERE: { constexpr int M = ACM_MODEL_DOUBLE_SPHERE; __VA_ARGS__; break; } \
                case ACM_MODEL_FOV: { constexpr int M = ACM_MODEL_FOV; __VA_ARGS__; break; }                     \
                default: return acm_fail(ctx, ACM_ERR_INVALID_ARG, "unknown camera model id %d", (int)(model));  \
            }                                                                                                    \
        } else return acm_fail(ctx, ACM_ERR_INVALID_ARG, "unknown residual kind %d", (int)(kind));              \
    } while (0)

static int32_t check_lin_args(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, const acm_points* uv) {
    ACM_REQUIRE(ctx, cam && xyz && uv, "linearize: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2, "linearize: xyz must have dim 3 and uv dim 2");
    ACM_REQUIRE(ctx, xyz->dtype == ACM_F64 && uv->dtype == ACM_F64, "linearize: f64 point buffers required");
    if (xyz->n != uv->n) return acm_fail(ctx, ACM_ERR_INVALID_PARAMS, "Number of 2D and 3D points must match");
    ACM_REQUIRE(ctx, cam->model >= 0 && cam->model <= 6 && cam->n_params == acm_n_params(cam->model), "linearize: bad camera block");
    return ACM_OK;
}

static bool peers_usable(const acm_ctx* ctx) { return ctx->peer_n > 1; }

// A peer exchange that timed out leaves the ranks' exchange counters out of step: refuse to go on
// until the host has re-attached the peers (acm_peer_detach + acm_peer_attach / acm_comm_init_all).
static int32_t check_peer_state(acm_ctx* ctx) {
    if (ctx->peer_failed)
        return acm_fail(ctx, ACM_ERR_PEER, "the NVLink peer exchange failed earlier (time-out or a peer's abort); detach and re-attach the peers");
    return ACM_OK;
}
static int32_t peer_failure(acm_ctx* ctx) {
    ctx->peer_failed = true;
    return acm_fail(ctx, ACM_ERR_PEER, "NVLink peer exchange timed out: a peer rank did not deliver its normal equations within ~2 s; "
                                       "every rank was aborted, detach and re-attach the peers before the next call");
}

// Enqueue one pass (+ the cross-rank sum).  With peers attached the sum happens inside the kernel;
// otherwise an NCCL all-reduce follows when a communicator is attached.  d_lm != nullptr: evaluate at
// the trial point of the device-resident LM state (NCCL path of acm_lm_solve).

// The exchange number that travels in the cells: the per-context counter in the low 48 bits (its parity picks the cell set) and a
// signature of the call (model, residual kind, one pass / solve) in the upper 16.  Ranks whose call sequences have drifted apart
// (one of them made a call the others did not) then wait for tags that never come and leave with ACM_ERR_PEER after the
// time-out, instead of silently adding the sums of different kernels.
static unsigned long long exchange_tag(unsigned long long seq, int model, int kind, int mode) {
    const unsigned long long sig = 0x8000ULL | ((unsigned long long)(mode & 3) << 8) | ((unsigned long long)(kind & 1) << 4) | (unsigned long long)(model & 15);
    return (seq & 0xFFFFFFFFFFFFULL) | (sig << 48);
}

static int32_t enqueue_linearize(acm_ctx* ctx, const acm_camera* cam, int32_t kind, LmState* d_lm, const acm_points* xyz,
                                 const acm_points* uv, double invalid_penalty, int* nacc) {
    LinKernelArgs a;
    memset(&a, 0, sizeof(a));
    make_lin_params(cam, &a.hp);
    a.lm = d_lm; a.mode = d_lm ? 1 : 0; a.max_passes = 1;
    a.pen2x2 = 2.0 * invalid_penalty * invalid_penalty;
    const bool use_peer = peers_usable(ctx) && !d_lm;
    if (use_peer) {
        int32_t rc = check_peer_state(ctx);
        if (rc) return rc;
        a.peer.bufs = ctx->d_peer_ptrs; a.peer.n_ranks = ctx->peer_n; a.peer.rank = ctx->peer_rank;
        a.peer.seq = exchange_tag(++ctx->peer_seq, cam->model, kind, 0);   // this launch executes exactly one exchange
    }
    ACM_DISPATCH_LIN(cam->model, kind, {
        int32_t rc = launch_lin<M, KIND>(ctx, a, xyz, uv);
        if (rc) return rc;
        *nacc = LinOps<M, KIND>::NACC;
    });
    if (!use_peer && ctx->comm && ctx->n_ranks > 1) return acm_allreduce_sum_f64(ctx, ctx->d_reduce, (size_t)*nacc);
    return ACM_OK;
}

static int32_t unpack_host(acm_ctx* ctx, const acm_camera* cam, int32_t kind, const double* r, acm_normal_equations* out) {
    memset(out, 0, sizeof(*out));
    out->n_params = cam->n_params;
    double cnt = 0.0;
    ACM_DISPATCH_LIN(cam->model, kind, (LinOps<M, KIND>::unpack(r, cam->params, out->H, out->g, &out->cost, &cnt)));
    out->n_valid = (uint64_t)cnt;
    return ACM_OK;
}

// host copy of the abort word of this rank's exchange buffer (only consulted when a result came back NaN)
static bool peer_abort_raised(acm_ctx* ctx) {
    unsigned long long w = 0;
    if (!ctx->peer_local) return false;
    if (cudaMemcpyAsync(&w, ctx->peer_local, sizeof(w), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return false;
    cudaStreamSynchronize(ctx->stream);
    return w != 0ULL;
}

extern "C" int32_t acm_linearize_async(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const acm_points* xyz, const acm_points* uv) {
    ACM_ENTER(ctx);
    int32_t rc = check_lin_args(ctx, cam, xyz, uv);
    if (rc) return rc;
    int nacc = 0;
    return enqueue_linearize(ctx, cam, residual_kind, nullptr, xyz, uv, 0.0, &nacc);
}

extern "C" int32_t acm_linearize(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const acm_points* xyz, const acm_points* uv,
                                 acm_normal_equations* out) {
    if (!ctx || !out) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    int32_t rc = check_lin_args(ctx, cam, xyz, uv);
    if (rc) return rc;
    int nacc = 0;
    rc = enqueue_linearize(ctx, cam, residual_kind, nullptr, xyz, uv, 0.0, &nacc);
    if (rc) return rc;
    ACM_CUDA(ctx, cudaMemcpyAsync(ctx->h_reduce, ctx->d_reduce, nacc * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (peers_usable(ctx)) {
        bool any_nan = false;
        for (int i = 0; i < nacc; ++i) any_nan = any_nan || !(ctx->h_reduce[i] == ctx->h_reduce[i]);
        if (any_nan && peer_abort_raised(ctx)) return peer_failure(ctx);
    }
    return unpack_host(ctx, cam, residual_kind, ctx->h_reduce, out);
}

extern "C" int32_t acm_linearize_host(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const double* xyz_aos, const double* uv_aos,
                                      size_t n, acm_normal_equations* out) {
    if (!ctx || !out) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_REQUIRE(ctx, cam && (n == 0 || (xyz_aos && uv_aos)), "linearize_host: null argument");
    // device buffers are kept between calls (grow-only): a 4 GB cudaMalloc/cudaFree pair per call
    // would cost more than the kernel
    if (ctx->cache_cap < n || !ctx->cache3) {
        cudaStreamSynchronize(ctx->stream);
        acm_points_destroy(ctx, ctx->cache3); acm_points_destroy(ctx, ctx->cache2);
        ctx->cache3 = ctx->cache2 = nullptr; ctx->cache_cap = 0;
        int32_t rc0 = acm_points_create(ctx, 3, n, ACM_F64, &ctx->cache3);
        if (!rc0) rc0 = acm_points_create(ctx, 2, n, ACM_F64, &ctx->cache2);
        if (rc0) { acm_points_destroy(ctx, ctx->cache3); ctx->cache3 = nullptr; return rc0; }
        ctx->cache_cap = n;
    }
    acm_points* xyz = ctx->cache3; acm_points* uv = ctx->cache2;
    xyz->n = n; uv->n = n;  // views of the first n points (the component stride is unchanged)
    int32_t rc = acm_points_upload_any(ctx, xyz, xyz_aos, n, 0);
    if (!rc) rc = acm_points_upload_any(ctx, uv, uv_aos, n, 0);
    if (!rc) rc = acm_linearize(ctx, cam, residual_kind, xyz, uv, out);
    cudaStreamSynchronize(ctx->stream);
    xyz->n = ctx->cache_cap; uv->n = ctx->cache_cap;
    return rc;
}

extern "C" int32_t acm_lm_default_config(acm_lm_config* cfg) {
    if (!cfg) return ACM_ERR_INVALID_ARG;
    cfg->max_iterations = 100;        // bin/camera_converter.rs:411
    cfg->cost_tolerance = 1e-6;       // :412
    cfg->parameter_tolerance = 1e-8;  // :413
    cfg->gradient_tolerance = 1e-6;   // :414
    cfg->lambda0 = 1e-3;
    cfg->invalid_penalty = 0.0;
    cfg->check_every = 4;
    return ACM_OK;
}

extern "C" int32_t acm_lm_solve(acm_ctx* ctx, const acm_camera* init, int32_t residual_kind, const acm_points* xyz, const acm_points* uv,
                                const double* lower, const double* upper, const acm_lm_config* cfg_in, double* out_params,
                                acm_lm_result* result) {
    if (!ctx || !out_params || !result) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    int32_t rc = check_lin_args(ctx, init, xyz, uv);
    if (rc) return rc;
    acm_lm_config cfg;
    if (cfg_in) cfg = *cfg_in; else acm_lm_default_config(&cfg);
    if (cfg.check_every < 1) cfg.check_every = 1;
    const auto t_start = std::chrono::steady_clock::now();
    const int P = init->n_params;
    LmState* h = static_cast<LmState*>(ctx->h_lm);
    LmState* d = static_cast<LmState*>(ctx->d_lm);
    memset(h, 0, sizeof(LmState));
    for (int i = 0; i < P; ++i) {
        h->lower[i] = lower ? lower[i] : -INFINITY;
        h->upper[i] = upper ? upper[i] : INFINITY;
        double v = init->params[i];
        v = v < h->lower[i] ? h->lower[i] : (v > h->upper[i] ? h->upper[i] : v);
        h->x[i] = v; h->xt[i] = v;
    }
    h->lambda = cfg.lambda0; h->nu = 2.0;
    h->cost_tol = cfg.cost_tolerance; h->param_tol = cfg.parameter_tolerance; h->grad_tol = cfg.gradient_tolerance;
    h->max_iter = cfg.max_iterations; h->first = 1; h->P = P; h->status = 3;
    const int max_passes = cfg.max_iterations + 2;
    const bool use_peer = peers_usable(ctx);
    const bool nccl_path = !use_peer && ctx->comm && ctx->n_ranks > 1;
    if (use_peer) { rc = check_peer_state(ctx); if (rc) return rc; }
    ACM_CUDA(ctx, cudaMemcpyAsync(d, h, sizeof(LmState), cudaMemcpyHostToDevice, ctx->stream));
    // the host copy doubles as the read-back buffer: wait until the upload has consumed it
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));

    double device_ms = 0.0;
    if (!nccl_path) {
        // the whole solve is ONE cooperative kernel: pass, reduction, NVLink exchange and LM step loop on the device
        LinKernelArgs a;
        memset(&a, 0, sizeof(a));
        make_lin_params(init, &a.hp);
        a.lm = d; a.mode = 2; a.max_passes = max_passes;
        a.pen2x2 = 2.0 * cfg.invalid_penalty * cfg.invalid_penalty;
        if (use_peer) {
            a.peer.bufs = ctx->d_peer_ptrs; a.peer.n_ranks = ctx->peer_n; a.peer.rank = ctx->peer_rank;
            a.peer.seq = exchange_tag(ctx->peer_seq + 1, init->model, residual_kind, 2);   // + pass inside the kernel
        }
        const bool want_trace = getenv("ACM_LM_TRACE") != nullptr;   // debug: per-phase clock64 stamps of block 0 -> stderr
        const size_t trace_words = (size_t)max_passes * 12 + (size_t)ctx->sm_count * 16 * 3;
        a.trace_pass = -1;
        if (want_trace) {
            rc = acm_ensure_scratch(ctx, trace_words * sizeof(long long));
            if (rc) return rc;
            ACM_CUDA(ctx, cudaMemsetAsync(ctx->d_scratch, 0, trace_words * sizeof(long long), ctx->stream));
            a.trace = static_cast<long long*>(ctx->d_scratch);
            if (atoi(getenv("ACM_LM_TRACE")) >= 2) a.trace_pass = getenv("ACM_LM_TRACE_PASS") ? atoi(getenv("ACM_LM_TRACE_PASS")) : 3;
        }
        ACM_DISPATCH_LIN(init->model, residual_kind, {
            rc = launch_lin<M, KIND>(ctx, a, xyz, uv);
            if (rc) return rc;
        });
        ACM_CUDA(ctx, cudaMemcpyAsync(h, d, sizeof(LmState), cudaMemcpyDeviceToHost, ctx->stream));
        ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (want_trace) {
            std::vector<long long> t(trace_words);
            ACM_CUDA(ctx, cudaMemcpy(t.data(), a.trace, t.size() * sizeof(long long), cudaMemcpyDeviceToHost));
            if (a.trace_pass >= 0) {
                // per-block skew of one pass: offsets (ns) from the earliest block's start
                const long long* q = &t[(size_t)max_passes * 12];
                long long t_min = 0;
                int nbk = 0;
                for (int b = 0; b < ctx->sm_count * 16 && q[3 * b]; ++b) { t_min = (b == 0 || q[3 * b] < t_min) ? q[3 * b] : t_min; nbk = b + 1; }
                for (int b = 0; b < nbk; ++b)
                    fprintf(stderr, "[acm lm skew] rank %d pass %d block %3d ns: start %lld  stream-end %lld  pass-end %lld\n", ctx->peer_rank, a.trace_pass, b,
                            q[3 * b] - t_min, q[3 * b + 1] - t_min, q[3 * b + 2] - t_min);
            }
            for (int k = 0; k < h->passes && k < max_passes; ++k) {
                const long long* q = &t[6 * k];
                fprintf(stderr, "[acm lm trace] rank %d pass %2d cycles: stream %lld  block-reduce %lld  reducers %lld  collect %lld  step %lld  | total %lld\n",
                        ctx->peer_rank, k, q[1] - q[0], q[2] - q[1], q[3] - q[2], q[4] - q[3], q[5] - q[4], q[5] - q[0]);
                const long long* u = &t[6 * (size_t)max_passes + 6 * k];
                if (u[0] && u[5])
                    fprintf(stderr, "[acm lm trace]          step cycles: unpack %lld  decide %lld  scale %lld  solve %lld  trial point %lld\n",
                            u[1] - u[0], u[2] - u[1], u[3] - u[2], u[4] - u[3], u[5] - u[4]);
            }
        }
        if (use_peer) ctx->peer_seq += (unsigned long long)h->passes;   // one exchange per executed pass, the same count on every rank
        device_ms = (double)(h->t_end_ns - h->t_begin_ns) * 1e-6;
        if (h->status == LM_STATUS_PEER_FAILURE) return peer_failure(ctx);
    } else {
        // NCCL path: one pass kernel + all-reduce + step kernel per iteration, `check_every` iterations enqueued blind
        int nacc = 0;
        int enq = 0;
        bool done = false;
        ACM_CUDA(ctx, cudaEventRecord(ctx->t0, ctx->stream));
        while (!done && enq < max_passes) {
            for (int k = 0; k < cfg.check_every && enq < max_passes; ++k, ++enq) {
                rc = enqueue_linearize(ctx, init, residual_kind, d, xyz, uv, cfg.invalid_penalty, &nacc);
                if (rc) return rc;
                ACM_DISPATCH_LIN(init->model, residual_kind, (lm_step_kernel<M, KIND><<<1, 128, 0, ctx->stream>>>(d, ctx->d_reduce)));
                ACM_CHECK_LAUNCH(ctx);
            }
            ACM_CUDA(ctx, cudaMemcpyAsync(h, d, sizeof(LmState), cudaMemcpyDeviceToHost, ctx->stream));
            ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            done = h->done != 0;
        }
        ACM_CUDA(ctx, cudaEventRecord(ctx->t1, ctx->stream));
        ACM_CUDA(ctx, cudaEventSynchronize(ctx->t1));
        float ms = 0.f;
        ACM_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->t0, ctx->t1));
        device_ms = ms;
    }
    for (int i = 0; i < P; ++i) out_params[i] = h->x[i];
    result->status = h->status; result->iterations = h->iterations; result->passes = h->passes;
    result->initial_cost = h->initial_cost; result->final_cost = h->cost; result->n_valid = (uint64_t)h->n_valid;
    result->elapsed_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    result->device_ms = device_ms;
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// project with `compute_jacobian = true` (README-era trait surface, reference README.md:119-126;
// per-model doc-comments double_sphere.rs:326-332 "2x6", kannala_brandt.rs:309-313 "2x8"):
// uv + the 2xP Jacobian w.r.t. [fx,fy,cx,cy,dist..], written as 2P rows of n doubles.
// ---------------------------------------------------------------------------------------
// Two points per thread: 16-byte loads of x, y, z, 16-byte streaming stores of u, v and of every Jacobian row (the rows are
// n doubles apart, so a row pair is 16-byte aligned whenever n is even and the base is); the odd tail and unaligned
// buffers go through the scalar form of the same body.
template <int M, int NV>
__global__ void __launch_bounds__(256) project_jacobian_kernel(const __grid_constant__ CamParams c, LinParams p, const double* __restrict__ X,
                                                               const double* __restrict__ Y, const double* __restrict__ Z,
                                                               double* __restrict__ U, double* __restrict__ V, double* __restrict__ J,
                                                               uint8_t* __restrict__ S, size_t n) {
    using LM_ = Lin<M, ACM_RESIDUAL_PIXEL>;
    constexpr int ND = LM_::ND, P = 4 + ND;
    const size_t npk = n / NV;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    auto one = [&](double x, double y, double z, double& u, double& v, double* row_u, double* row_v) -> int {
        int st = CamModel<M>::template project<false>(c, x, y, z, u, v);
        double ru, rv, au[2 + ND], av[2 + ND];
#pragma unroll
        for (int k = 0; k < P; ++k) row_u[k] = row_v[k] = 0.0;
        if (st == ACM_POINT_OK && LM_::eval(p, x, y, z, 0.0, 0.0, ru, rv, au, av)) {
            row_u[0] = au[0]; row_u[2] = 1.0; row_v[1] = av[0]; row_v[3] = 1.0;
#pragma unroll
            for (int k = 0; k < ND; ++k) { row_u[4 + k] = au[2 + k]; row_v[4 + k] = av[2 + k]; }
        } else {
            if (st == ACM_POINT_OK) st = ACM_POINT_NUMERICAL_ERROR;
            u = v = acm_nan();
        }
        return st;
    };
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npk; i += stride) {
        if constexpr (NV == 2) {
            const double2 x = __ldcs(reinterpret_cast<const double2*>(X) + i), y = __ldcs(reinterpret_cast<const double2*>(Y) + i),
                          z = __ldcs(reinterpret_cast<const double2*>(Z) + i);
            double u0, v0, u1, v1, ru0[P], rv0[P], ru1[P], rv1[P];
            const int s0 = one(x.x, y.x, z.x, u0, v0, ru0, rv0), s1 = one(x.y, y.y, z.y, u1, v1, ru1, rv1);
            __stcs(reinterpret_cast<double2*>(U) + i, make_double2(u0, u1));
            __stcs(reinterpret_cast<double2*>(V) + i, make_double2(v0, v1));
            if (S) __stcs(reinterpret_cast<uchar2*>(S) + i, make_uchar2((uint8_t)s0, (uint8_t)s1));
#pragma unroll
            for (int k = 0; k < P; ++k) {
                __stcs(reinterpret_cast<double2*>(J + (size_t)k * n) + i, make_double2(ru0[k], ru1[k]));
                __stcs(reinterpret_cast<double2*>(J + (size_t)(P + k) * n) + i, make_double2(rv0[k], rv1[k]));
            }
        } else {
            double u, v, row_u[P], row_v[P];
            const int st = one(X[i], Y[i], Z[i], u, v, row_u, row_v);
            U[i] = u; V[i] = v;
            if (S) S[i] = (uint8_t)st;
#pragma unroll
            for (int k = 0; k < P; ++k) { J[(size_t)k * n + i] = row_u[k]; J[(size_t)(P + k) * n + i] = row_v[k]; }
        }
    }
}

extern "C" int32_t acm_project_jacobian(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, double* d_jac,
                                        uint8_t* d_status) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv && d_jac, "project_jacobian: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2 && xyz->n == uv->n, "project_jacobian: shape mismatch");
    ACM_REQUIRE(ctx, xyz->dtype == ACM_F64 && uv->dtype == ACM_F64, "project_jacobian: f64 buffers required");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    LinParams p;
    make_lin_params(cam, &p);
    const size_t n = xyz->n;
    if (n == 0) return ACM_OK;
    const bool vec = (n % 2 == 0) && ((reinterpret_cast<uintptr_t>(d_jac) & 15) == 0) && (!d_status || (reinterpret_cast<uintptr_t>(d_status) & 1) == 0);
    if (vec) {
        const int grid = grid_for(ctx, n / 2, 256, 4);
        ACM_DISPATCH_MODEL(cam->model, (project_jacobian_kernel<M, 2><<<grid, 256, 0, ctx->stream>>>(
            c, p, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), comp<double>(uv, 0), comp<double>(uv, 1), d_jac, d_status, n)))
    } else {
        const int grid = grid_for(ctx, n, 256, 4);
        ACM_DISPATCH_MODEL(cam->model, (project_jacobian_kernel<M, 1><<<grid, 256, 0, ctx->stream>>>(
            c, p, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), comp<double>(uv, 0), comp<double>(uv, 1), d_jac, d_status, n)))
    }
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// project with the 2x3 Jacobian w.r.t. the 3-D point (the other reading of the README-era
// `compute_jacobian` flag: trait doc reference src/camera/mod.rs:246-252 "Jacobian matrix (2x3)").
// uv + six rows of n doubles: du/dx, du/dy, du/dz, dv/dx, dv/dy, dv/dz.
// ---------------------------------------------------------------------------------------
template <int M, int NV>
__global__ void __launch_bounds__(256) project_point_jacobian_kernel(const __grid_constant__ CamParams c, LinParams p, const double* __restrict__ X,
                                                                     const double* __restrict__ Y, const double* __restrict__ Z,
                                                                     double* __restrict__ U, double* __restrict__ V, double* __restrict__ J,
                                                                     uint8_t* __restrict__ S, size_t n) {
    const size_t npk = n / NV;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    auto one = [&](double x, double y, double z, double& u, double& v, double* ju, double* jv) -> int {
        const int st = CamModel<M>::template project<false>(c, x, y, z, u, v);
        if (st == ACM_POINT_OK) PointJac<M>::eval(p, x, y, z, ju, jv);
        else { u = v = acm_nan(); ju[0] = ju[1] = ju[2] = jv[0] = jv[1] = jv[2] = 0.0; }
        return st;
    };
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npk; i += stride) {
        if constexpr (NV == 2) {
            const double2 x = __ldcs(reinterpret_cast<const double2*>(X) + i), y = __ldcs(reinterpret_cast<const double2*>(Y) + i),
                          z = __ldcs(reinterpret_cast<const double2*>(Z) + i);
            double u0, v0, u1, v1, ju0[3], jv0[3], ju1[3], jv1[3];
            const int s0 = one(x.x, y.x, z.x, u0, v0, ju0, jv0), s1 = one(x.y, y.y, z.y, u1, v1, ju1, jv1);
            __stcs(reinterpret_cast<double2*>(U) + i, make_double2(u0, u1));
            __stcs(reinterpret_cast<double2*>(V) + i, make_double2(v0, v1));
            if (S) __stcs(reinterpret_cast<uchar2*>(S) + i, make_uchar2((uint8_t)s0, (uint8_t)s1));
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                __stcs(reinterpret_cast<double2*>(J + (size_t)k * n) + i, make_double2(ju0[k], ju1[k]));
                __stcs(reinterpret_cast<double2*>(J + (size_t)(3 + k) * n) + i, make_double2(jv0[k], jv1[k]));
            }
        } else {
            double u, v, ju[3], jv[3];
            const int st = one(X[i], Y[i], Z[i], u, v, ju, jv);
            U[i] = u; V[i] = v;
            if (S) S[i] = (uint8_t)st;
#pragma unroll
            for (int k = 0; k < 3; ++k) { __stcs(J + (size_t)k * n + i, ju[k]); __stcs(J + (size_t)(3 + k) * n + i, jv[k]); }
        }
    }
}

extern "C" int32_t acm_project_point_jacobian(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, double* d_jac,
                                              uint8_t* d_status) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv && d_jac, "project_point_jacobian: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2 && xyz->n == uv->n, "project_point_jacobian: shape mismatch");
    ACM_REQUIRE(ctx, xyz->dtype == ACM_F64 && uv->dtype == ACM_F64, "project_point_jacobian: f64 buffers required");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    LinParams p;
    make_lin_params(cam, &p);
    const size_t n = xyz->n;
    if (n == 0) return ACM_OK;
    const bool vec = (n % 2 == 0) && ((reinterpret_cast<uintptr_t>(d_jac) & 15) == 0) && (!d_status || (reinterpret_cast<uintptr_t>(d_status) & 1) == 0);
    if (vec) {
        const int grid = grid_for(ctx, n / 2, 256, 4);
        ACM_DISPATCH_MODEL(cam->model, (project_point_jacobian_kernel<M, 2><<<grid, 256, 0, ctx->stream>>>(
            c, p, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), comp<double>(uv, 0), comp<double>(uv, 1), d_jac, d_status, n)))
    } else {
        const int grid = grid_for(ctx, n, 256, 4);
        ACM_DISPATCH_MODEL(cam->model, (project_point_jacobian_kernel<M, 1><<<grid, 256, 0, ctx->stream>>>(
            c, p, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), comp<double>(uv, 0), comp<double>(uv, 1), d_jac, d_status, n)))
    }
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}
