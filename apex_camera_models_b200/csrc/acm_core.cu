// Context, memory, point buffers (AoS <-> SoA), camera parameter blocks, NCCL plumbing.
#include <dlfcn.h>

#include <atomic>
#include <chrono>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <cmath>

#include <new>

#include "acm_internal.cuh"

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

void acm_set_global_error(const char* msg) { g_last_error = msg; }

int32_t acm_fail(acm_ctx* ctx, int32_t code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    g_last_error = buf;
    return code;
}

extern "C" const char* acm_last_error(const acm_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }
extern "C" int32_t acm_abi_version(void) { return ACM_ABI_VERSION; }

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
extern "C" int32_t acm_ctx_create(int32_t device, void* cuda_stream, acm_ctx** out) {
    if (!out) return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "acm_ctx_create: null output");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return acm_fail(nullptr, ACM_ERR_NO_DEVICE, "no CUDA device available (%s); libacm has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "device %d out of range [0,%d)", device, count);
    acm_ctx* ctx = new (std::nothrow) acm_ctx();
    if (!ctx) return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "out of host memory");
    ctx->device = device;
    ctx->comm = nullptr; ctx->n_ranks = 1; ctx->rank = 0;
    ctx->launches = 0;
    ctx->d_partials = nullptr; ctx->partials_cap = 0; ctx->d_reduce = nullptr; ctx->d_ticket = nullptr; ctx->h_reduce = nullptr;
    ctx->d_lm = nullptr; ctx->h_lm = nullptr; ctx->d_stage[0] = ctx->d_stage[1] = nullptr; ctx->stage_cap = 0;
    ctx->h_stage = nullptr; ctx->h_stage_cap = 0;
    ctx->cache3 = nullptr; ctx->cache2 = nullptr; ctx->cache_cap = 0;
    ctx->d_scratch = nullptr; ctx->scratch_cap = 0;
    for (int i = 0; i < ACM_FREE_LIST; ++i) { ctx->free_ptr[i] = nullptr; ctx->free_bytes[i] = 0; }
    ctx->peer_local = nullptr; ctx->d_peer_ptrs = nullptr; ctx->peer_n = 0; ctx->peer_rank = 0; ctx->peer_seq = 0; ctx->peer_failed = false;
    ctx->group = nullptr; ctx->lm_tag = 0; ctx->d_lm_ll = nullptr; ctx->lm_ll_cap = 0; ctx->coop_launch = 0;
    ctx->h_small = nullptr; ctx->d_small_alias = nullptr; ctx->small_cap = 0;
    ctx->cam_cache_valid = false;
    for (int i = 0; i < ACM_MAX_PEERS; ++i) ctx->peer_mapped[i] = nullptr;
#define CREATE_CUDA(call)                                                                                     \
    do { cudaError_t _e = (call); if (_e != cudaSuccess) { int32_t rc = acm_fail(nullptr, ACM_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); delete ctx; return rc; } } while (0)
    CREATE_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CREATE_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    ctx->cc = prop.major * 10 + prop.minor;
    CREATE_CUDA(cudaDeviceGetAttribute(&ctx->coop_launch, cudaDevAttrCooperativeLaunch, device));
    if (cuda_stream) { ctx->stream = (cudaStream_t)cuda_stream; ctx->owns_stream = false; }
    else { CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->owns_stream = true; }
    CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaEventCreate(&ctx->t0));
    CREATE_CUDA(cudaEventCreate(&ctx->t1));
    for (int i = 0; i < 4; ++i) CREATE_CUDA(cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming));
    CREATE_CUDA(cudaMalloc(&ctx->d_reduce, 2048 * sizeof(double)));
    CREATE_CUDA(cudaMalloc(&ctx->d_ticket, 64 * sizeof(unsigned int)));
    CREATE_CUDA(cudaMemset(ctx->d_ticket, 0, 64 * sizeof(unsigned int)));
    CREATE_CUDA(cudaMallocHost(&ctx->h_reduce, 2048 * sizeof(double)));
    CREATE_CUDA(cudaMalloc(&ctx->d_lm, 4096));
    CREATE_CUDA(cudaMemset(ctx->d_lm, 0, 4096));
    CREATE_CUDA(cudaMallocHost(&ctx->h_lm, 4096));
#undef CREATE_CUDA
    *out = ctx;
    return ACM_OK;
}

static void acm_free_list_release(acm_ctx* ctx) {
    for (int i = 0; i < ACM_FREE_LIST; ++i) {
        if (ctx->free_ptr[i]) cudaFree(ctx->free_ptr[i]);
        ctx->free_ptr[i] = nullptr; ctx->free_bytes[i] = 0;
    }
}

int32_t acm_device_malloc(acm_ctx* ctx, void** out, size_t bytes) {
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        acm_free_list_release(ctx);
        e = cudaMalloc(out, bytes ? bytes : 1);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return acm_fail(ctx, ACM_ERR_CUDA, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    return ACM_OK;
}

extern "C" int32_t acm_ctx_destroy(acm_ctx* ctx) {
    if (!ctx) return ACM_OK;
    if (ctx->group) acm_group_dissolve(ctx);  // stops the group's workers and detaches every member (acm_multi.cu)
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    acm_comm_destroy(ctx);
    acm_peer_detach(ctx);
    acm_points_destroy(ctx, ctx->cache3); acm_points_destroy(ctx, ctx->cache2);
    acm_free_list_release(ctx);
    cudaFree(ctx->peer_local);
    cudaFree(ctx->d_lm_ll);
    cudaFreeHost(ctx->h_small);
    cudaFree(ctx->d_scratch);
    cudaFree(ctx->d_partials); cudaFree(ctx->d_reduce); cudaFree(ctx->d_ticket); cudaFreeHost(ctx->h_reduce);
    cudaFree(ctx->d_lm); cudaFreeHost(ctx->h_lm);
    cudaFree(ctx->d_stage[0]); cudaFree(ctx->d_stage[1]); cudaFreeHost(ctx->h_stage);
    for (int i = 0; i < 4; ++i) cudaEventDestroy(ctx->chunk_ev[i]);
    cudaEventDestroy(ctx->t0); cudaEventDestroy(ctx->t1);
    cudaStreamDestroy(ctx->copy_stream);
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return ACM_OK;
}

extern "C" int32_t acm_ctx_sync(acm_ctx* ctx) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ACM_OK;
}

extern "C" int32_t acm_ctx_device_info(const acm_ctx* ctx, int64_t info[4]) {
    if (!ctx || !info) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    info[0] = ctx->sm_count; info[1] = (int64_t)ctx->l2_bytes; info[2] = 0; info[3] = ctx->cc;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess) info[2] = (int64_t)prop.sharedMemPerBlockOptin;
    return ACM_OK;
}

extern "C" int32_t acm_timer_start(acm_ctx* ctx) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaEventRecord(ctx->t0, ctx->stream));
    return ACM_OK;
}
extern "C" int32_t acm_timer_stop(acm_ctx* ctx, float* elapsed_ms) {
    if (!ctx || !elapsed_ms) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_CUDA(ctx, cudaEventRecord(ctx->t1, ctx->stream));
    ACM_CUDA(ctx, cudaEventSynchronize(ctx->t1));
    ACM_CUDA(ctx, cudaEventElapsedTime(elapsed_ms, ctx->t0, ctx->t1));
    return ACM_OK;
}
extern "C" uint64_t acm_ctx_kernel_launches(const acm_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------------------------------
// camera parameter blocks (host logic; mirrors `new` and `validate_params` of every model)
// ---------------------------------------------------------------------------------------
static const int kNParams[7] = {4, 9, 8, 5, 6, 6, 5};
static const char* kExpect[7] = {
    "Expected 4 parameters (fx, fy, cx, cy), got %zu",                      // pinhole.rs:82-87
    "Expected 9 parameters (fx, fy, cx, cy, k1, k2, p1, p2, k3), got %zu",  // rad_tan.rs:108-113
    "Expected 8 parameters, got %zu",                                       // kannala_brandt.rs:123-128
    "Expected 5 parameters (fx, fy, cx, cy, alpha), got %zu",               // ucm.rs:114-119
    "Expected 6 parameters (fx, fy, cx, cy, alpha, beta), got %zu",         // eucm.rs
    "Expected 6 parameters (fx, fy, cx, cy, alpha, xi), got %zu",           // double_sphere.rs:134-139
    "Expected 5 parameters (fx, fy, cx, cy, w), got %zu"};                  // fov.rs:114-119

extern "C" int32_t acm_n_params(int32_t model) { return (model >= 0 && model < 7) ? kNParams[model] : ACM_ERR_INVALID_ARG; }

static void put_msg(char* msg, size_t len, const char* text) {
    if (msg && len) { strncpy(msg, text, len - 1); msg[len - 1] = 0; }
}

extern "C" int32_t acm_validate_params(const acm_camera* cam, char* msg, size_t msg_len) {
    put_msg(msg, msg_len, "");
    if (!cam || cam->model < 0 || cam->model > 6 || cam->n_params != kNParams[cam->model]) {
        put_msg(msg, msg_len, "invalid camera block");
        return ACM_ERR_INVALID_ARG;
    }
    const double* p = cam->params;
    // validation::validate_intrinsics (mod.rs:362-370)
    if (p[0] <= 0.0 || p[1] <= 0.0) { put_msg(msg, msg_len, "Focal length must be positive"); return ACM_ERR_FOCAL_LENGTH; }
    if (!isfinite(p[2]) || !isfinite(p[3])) { put_msg(msg, msg_len, "Principal point must be finite"); return ACM_ERR_PRINCIPAL_POINT; }
    char buf[128];
    switch (cam->model) {
        case ACM_MODEL_UCM:  // ucm.rs:467-477
            if (!isfinite(p[4])) { put_msg(msg, msg_len, "alpha must be finite"); return ACM_ERR_INVALID_PARAMS; }
            break;
        case ACM_MODEL_EUCM:  // eucm.rs:501-517
            if (!isfinite(p[4])) { put_msg(msg, msg_len, "alpha must be finite"); return ACM_ERR_INVALID_PARAMS; }
            if (!isfinite(p[5])) { put_msg(msg, msg_len, "beta must be finite"); return ACM_ERR_INVALID_PARAMS; }
            break;
        case ACM_MODEL_DOUBLE_SPHERE:  // double_sphere.rs:592-608
            if (p[4] <= 0.0 || p[4] > 1.0) { put_msg(msg, msg_len, "alpha must be in (0, 1]"); return ACM_ERR_INVALID_PARAMS; }
            if (!isfinite(p[5])) { put_msg(msg, msg_len, "xi must be finite"); return ACM_ERR_INVALID_PARAMS; }
            break;
        case ACM_MODEL_FOV:  // fov.rs:457-468
            if (!isfinite(p[4]) || p[4] <= 2.220446049250313e-16 || p[4] > 3.0) {
                snprintf(buf, sizeof(buf), "w must be in range (epsilon, 3.0], got %g", p[4]);
                put_msg(msg, msg_len, buf);
                return ACM_ERR_INVALID_PARAMS;
            }
            break;
        default: break;  // pinhole / rad_tan / kannala_brandt: intrinsics only
    }
    return ACM_OK;
}

extern "C" int32_t acm_camera_new(int32_t model, const double* params, size_t n, acm_camera* out, char* msg, size_t msg_len) {
    put_msg(msg, msg_len, "");
    if (!out || model < 0 || model > 6 || (!params && n)) { put_msg(msg, msg_len, "invalid argument"); return ACM_ERR_INVALID_ARG; }
    if ((int)n != kNParams[model]) {
        char buf[128];
        snprintf(buf, sizeof(buf), kExpect[model], n);
        put_msg(msg, msg_len, buf);
        return ACM_ERR_INVALID_PARAMS;
    }
    memset(out, 0, sizeof(*out));
    out->model = model; out->width = 0; out->height = 0; out->n_params = (int32_t)n;
    for (size_t i = 0; i < n; ++i) out->params[i] = params[i];
    // only Pinhole and RadTan validate inside `new` (pinhole.rs:101, rad_tan.rs:135)
    if (model == ACM_MODEL_PINHOLE || model == ACM_MODEL_RADTAN) return acm_validate_params(out, msg, msg_len);
    return ACM_OK;
}

static int32_t make_cam_params_uncached(acm_ctx* ctx, const acm_camera* cam, CamParams* c);

// The host-side gates of the contracted Newton iterations (Kannala-Brandt, RadTan) cost 20-100 us; a context remembers the
// block of the last camera it prepared, so that a loop of scalar project / unproject calls on one model pays them once.
int32_t acm_make_cam_params(acm_ctx* ctx, const acm_camera* cam, CamParams* c) {
    if (ctx && cam && ctx->cam_cache_valid && cam->model == ctx->cam_cache_key.model && cam->width == ctx->cam_cache_key.width &&
        cam->height == ctx->cam_cache_key.height && cam->n_params == ctx->cam_cache_key.n_params && cam->n_params >= 0 &&
        cam->n_params <= ACM_MAX_PARAMS && memcmp(cam->params, ctx->cam_cache_key.params, sizeof(double) * cam->n_params) == 0) {
        *c = ctx->cam_cache_val;
        return ACM_OK;
    }
    int32_t rc = make_cam_params_uncached(ctx, cam, c);
    if (rc == ACM_OK && ctx) { ctx->cam_cache_key = *cam; ctx->cam_cache_val = *c; ctx->cam_cache_valid = true; }
    return rc;
}

static int32_t make_cam_params_uncached(acm_ctx* ctx, const acm_camera* cam, CamParams* c) {
    if (!cam || cam->model < 0 || cam->model > 6) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "invalid camera model id");
    if (cam->n_params != kNParams[cam->model])
        return acm_fail(ctx, ACM_ERR_INVALID_PARAMS, "model %d expects %d parameters, got %d", cam->model, kNParams[cam->model], cam->n_params);
    memset(c, 0, sizeof(*c));
    c->fx = cam->params[0]; c->fy = cam->params[1]; c->cx = cam->params[2]; c->cy = cam->params[3];
    for (int i = 4; i < cam->n_params; ++i) c->d[i - 4] = cam->params[i];
    c->W = (double)cam->width; c->H = (double)cam->height;
    c->has_resolution = (cam->width > 0 && cam->height > 0) ? 1 : 0;
    c->model = cam->model;
    {   // reciprocals for the exact division by the (kernel-invariant) focal lengths, see acm_div_by()
        volatile double one = 1.0, fx = c->fx, fy = c->fy;
        c->ifx = one / fx; c->ify = one / fy;
        int ex = 0, ey = 0;
        const bool okx = std::isnormal(c->fx) && (frexp(c->fx, &ex), ex >= -99 && ex <= 101);
        const bool oky = std::isnormal(c->fy) && (frexp(c->fy, &ey), ey >= -99 && ey <= 101);
        c->fast_div = (okx && oky) ? 1 : 0;
    }
    // per-model constants, in the reference's operation order (volatile: no host-side contraction)
    volatile double alpha = c->d[0];
    switch (cam->model) {
        case ACM_MODEL_UCM: {  // ucm.rs:154-161, :177-184, :346-347
            volatile double gamma = 1.0 - alpha;
            c->k0 = (alpha <= 0.5) ? alpha / (1.0 - alpha) : (1.0 - alpha) / alpha;
            volatile double g2 = gamma * gamma;
            volatile double den = 2.0 * alpha - 1.0;
            c->k1 = g2 / den;
            c->k2 = alpha / gamma;
            break;
        }
        case ACM_MODEL_EUCM: {  // eucm.rs:171, :196
            volatile double beta = c->d[1];
            volatile double t = 2.0 * alpha - 1.0;
            c->k0 = (alpha - 1.0) / t;
            volatile double ib = 1.0 / beta;
            c->k1 = ib * t;
            break;
        }
        case ACM_MODEL_DOUBLE_SPHERE: {  // double_sphere.rs:177-184, :204
            volatile double xi = c->d[1];
            volatile double w1 = (alpha <= 0.5) ? alpha / (1.0 - alpha) : (1.0 - alpha) / alpha;
            volatile double a = 2.0 * w1;
            volatile double b = a * xi;
            volatile double cc = xi * xi;
            volatile double s = b + cc;
            volatile double s1 = s + 1.0;
            c->k0 = (w1 + xi) / sqrt(s1);
            volatile double t = 2.0 * alpha - 1.0;
            c->k1 = 1.0 / t;
            break;
        }
        case ACM_MODEL_KANNALA_BRANDT: {
            // unproject solves g(theta) = theta (1 + k1 theta^2 + .. + k4 theta^8) = ru by Newton from theta0 = ru, ru in
            // (1e-6, pi/2] (kannala_brandt.rs:470-520).  Kantorovich on |theta| <= tb: with m <= g', |g''| <= Mb and the first
            // step bounded by eta = max|g(ru) - ru| / m, h = Mb eta / m <= 0.4 guarantees quadratic convergence inside a ball of
            // radius eta (1 - sqrt(1 - 2h)) / h around theta0, for every ru.  The reference's loop (10 iterations, stop at
            // |delta| < 1e-6, fail on |g'| < EPS) then returns Ok for every pixel and its iterate is within (Mb/2m) 1e-12 of the
            // root -- which lets the batch kernel run a contracted (FMA + reciprocal) Newton: same status, theta within 1e-11.
            // Cameras that fail the test keep the IEEE loop.
            // m, Mb and max|g(ru) - ru| are bounded rigorously from 1024 samples plus a Lipschitz margin taken from
            // absolute-value bounds of the next derivative (the sample camera has k3 < 0, which makes plain |k| bounds useless).
            const double tb = 1.75, rmax = 3.14159265358979323846 / 2.0;
            const double k[4] = {c->d[0], c->d[1], c->d[2], c->d[3]};
            double L1 = 0.0, L2 = 0.0, L3 = 0.0;   // bounds of |g1 - 1|, |g2|, |g3| (first to third derivative of g) from |k_i|
            for (int i = 0; i < 4; ++i) {
                const int p = 2 * (i + 1);   // term k_i theta^(p+1)
                L1 += (p + 1) * fabs(k[i]) * pow(tb, p);
                L2 += (p + 1) * p * fabs(k[i]) * pow(tb, p - 1);
                L3 += (p + 1) * p * (p - 1) * fabs(k[i]) * pow(tb, p - 2);
            }
            c->fast_newton = 0;
            if (std::isfinite(L3) && L3 < 1e6) {
                const int NS = 1024;
                const double dt = tb / NS;
                double gmin = INFINITY, g2max = 0.0, f0max = 0.0;
                for (int j = 0; j <= NS; ++j) {
                    const double t = j * dt, t2 = t * t;
                    const double gp = 1.0 + t2 * (3.0 * k[0] + t2 * (5.0 * k[1] + t2 * (7.0 * k[2] + t2 * 9.0 * k[3])));
                    const double gpp = t * (6.0 * k[0] + t2 * (20.0 * k[1] + t2 * (42.0 * k[2] + t2 * 72.0 * k[3])));
                    gmin = fmin(gmin, gp); g2max = fmax(g2max, fabs(gpp));
                    if (t <= rmax + dt) f0max = fmax(f0max, fabs(t * t2 * (k[0] + t2 * (k[1] + t2 * (k[2] + t2 * k[3])))));
                }
                const double m = gmin - L2 * dt, Mb = g2max + L3 * dt, F0 = f0max + L1 * dt;
                if (m >= 0.5) {
                    const double eta = F0 / m, h = Mb * eta / m;
                    const double radius = h > 1e-12 ? eta * (1.0 - sqrt(1.0 - 2.0 * fmin(h, 0.5))) / h : eta;
                    if (h <= 0.4 && radius <= tb - rmax && Mb / (2.0 * m) <= 4.0) c->fast_newton = 1;
                }
            }
            break;
        }
        case ACM_MODEL_RADTAN: {
            // Gate of the contracted 2-D Newton iteration of unproject (acm_models.cuh: unproject_newton_fast).  The kernel
            // itself is safe for any camera -- every decision it cannot take with a margin goes back to the IEEE loop -- so
            // the gate only has to keep out cameras for which that would be the common case or for which a perturbation of
            // a few 1e-15 in an iterate could grow: the reference's own loop is run here (plain IEEE doubles) on a 25 x 25
            // grid of targets covering the image (the bounds test admits no other pixel) and must stop within 12 steps
            // everywhere with a Jacobian that is nowhere near singular (|det| >= 0.05 (|j00 j11| + |j10 j01|)) and steps
            // that shrink (no step larger than the first one).  Sane calibrations (the sample camera: 3 evaluations, det ~ 1)
            // pass; strong barrel distortion whose mapping folds over inside the image does not and keeps the IEEE loop.
            c->fast_newton = 0;
            const double k1 = c->d[0], k2 = c->d[1], p1 = c->d[2], p2 = c->d[3], k3 = c->d[4];
            bool ok = c->has_resolution && c->fast_div && std::isfinite(k1) && std::isfinite(k2) && std::isfinite(k3) && std::isfinite(p1) &&
                      std::isfinite(p2) && std::isfinite(c->cx) && std::isfinite(c->cy);
            const int G = 24;
            for (int gy = 0; ok && gy <= G; ++gy) {
                for (int gx = 0; ok && gx <= G; ++gx) {
                    const double tx = (c->W * gx / G - c->cx) / c->fx, ty = (c->H * gy / G - c->cy) / c->fy;
                    if (!(fabs(tx) <= 50.0 && fabs(ty) <= 50.0)) { ok = false; break; }
                    double px = tx, py = ty, first = -1.0;
                    bool stopped = false;
                    for (int it = 0; it < 12 && !stopped; ++it) {
                        const double x = px, y = py, r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2;
                        const double rad = 1.0 + k1 * r2 + k2 * r4 + k3 * r6;
                        const double ex = x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x) - tx;
                        const double ey = y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y - ty;
                        if (sqrt(ex * ex + ey * ey) < 1e-6) { stopped = true; break; }
                        const double common = k1 + 2.0 * k2 * r2 + 3.0 * k3 * r4;
                        const double j00 = rad + x * common * 2.0 * x + 2.0 * p1 * y + p2 * 6.0 * x, j01 = x * common * 2.0 * y + 2.0 * p1 * x + p2 * 2.0 * y;
                        const double j10 = y * common * 2.0 * x + p1 * 2.0 * x + 2.0 * p2 * y, j11 = rad + y * common * 2.0 * y + p1 * 6.0 * y + 2.0 * p2 * x;
                        const double det = j00 * j11 - j10 * j01;
                        if (!(fabs(det) >= 0.05 * (fabs(j00 * j11) + fabs(j10 * j01)))) { ok = false; break; }
                        const double dx = (j11 * ex - j01 * ey) / det, dy = (j00 * ey - j10 * ex) / det;
                        const double step = sqrt(dx * dx + dy * dy);
                        if (first < 0.0) first = step;
                        if (!(step <= first)) { ok = false; break; }
                        px -= dx; py -= dy;
                        if (step < 1e-6) stopped = true;
                    }
                    if (!stopped) ok = false;
                }
            }
            c->fast_newton = ok ? 1 : 0;
            break;
        }
        case ACM_MODEL_FOV: {  // fov.rs:296, :340
            c->k0 = tan(c->d[0] / 2.0);
            break;
        }
        default: break;
    }
    return ACM_OK;
}

// 1 when acm_unproject runs the contracted Newton iteration for this camera (Kannala-Brandt cameras that pass the
// host-side convergence proof above, RadTan cameras that pass the grid gate), 0 when it keeps the IEEE loop; negative on
// an invalid camera block
extern "C" int32_t acm_camera_fast_unproject(const acm_camera* cam) {
    CamParams c;
    int32_t rc = acm_make_cam_params(nullptr, cam, &c);
    if (rc) return rc;
    return ((c.model == ACM_MODEL_KANNALA_BRANDT || c.model == ACM_MODEL_RADTAN) && c.fast_newton) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------
// raw memory
// ---------------------------------------------------------------------------------------
extern "C" int32_t acm_device_alloc(acm_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_CUDA(ctx, cudaSetDevice(ctx->device));
    { int32_t rc = acm_device_malloc(ctx, out, bytes); if (rc) return rc; }
    return ACM_OK;
}
extern "C" int32_t acm_device_free(acm_ctx* ctx, void* p) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaFree(p));
    return ACM_OK;
}
extern "C" int32_t acm_host_alloc_pinned(acm_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_CUDA(ctx, cudaSetDevice(ctx->device));
    ACM_CUDA(ctx, cudaMallocHost(out, bytes ? bytes : 1));
    return ACM_OK;
}
extern "C" int32_t acm_host_free_pinned(acm_ctx* ctx, void* p) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaFreeHost(p));
    return ACM_OK;
}
extern "C" int32_t acm_memcpy_h2d(acm_ctx* ctx, void* dst, const void* src, size_t bytes) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return ACM_OK;
}
extern "C" int32_t acm_memcpy_d2h(acm_ctx* ctx, void* dst, const void* src, size_t bytes) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return ACM_OK;
}
extern "C" int32_t acm_memcpy_d2d(acm_ctx* ctx, void* dst, const void* src, size_t bytes) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return ACM_OK;
}
extern "C" int32_t acm_memset_d(acm_ctx* ctx, void* dst, int value, size_t bytes) {
    ACM_ENTER(ctx);
    ACM_CUDA(ctx, cudaMemsetAsync(dst, value, bytes, ctx->stream));
    return ACM_OK;
}

int32_t acm_ensure_stage(acm_ctx* ctx, size_t bytes) {
    if (ctx->stage_cap >= bytes) return ACM_OK;
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    for (int i = 0; i < 2; ++i) { cudaFree(ctx->d_stage[i]); ctx->d_stage[i] = nullptr; }
    ctx->stage_cap = 0;
    for (int i = 0; i < 2; ++i) ACM_CUDA(ctx, cudaMalloc(&ctx->d_stage[i], bytes));
    ctx->stage_cap = bytes;
    return ACM_OK;
}

int32_t acm_ensure_host_stage(acm_ctx* ctx, size_t bytes) {
    if (ctx->h_stage_cap >= bytes) return ACM_OK;
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFreeHost(ctx->h_stage); ctx->h_stage = nullptr; ctx->h_stage_cap = 0;
    ACM_CUDA(ctx, cudaMallocHost(&ctx->h_stage, bytes));
    ctx->h_stage_cap = bytes;
    return ACM_OK;
}

int32_t acm_ensure_scratch(acm_ctx* ctx, size_t bytes) {
    if (ctx->scratch_cap >= bytes) return ACM_OK;
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->d_scratch); ctx->d_scratch = nullptr; ctx->scratch_cap = 0;
    const size_t want = bytes + bytes / 4;  // head room: the arena only ever grows
    { int32_t rc = acm_device_malloc(ctx, &ctx->d_scratch, want); if (rc) return rc; }
    ctx->scratch_cap = want;
    return ACM_OK;
}

int32_t acm_kernel_blocks_per_sm(acm_ctx* ctx, const void* fn, int block, size_t smem, int* out) {
    auto it = ctx->blocks_per_sm.find(fn);
    if (it != ctx->blocks_per_sm.end()) { *out = it->second; return ACM_OK; }
    // both the opt-in and the occupancy are properties of (kernel, device): cached per context, not per process
    if (smem > 48 * 1024) ACM_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int b = 0;
    ACM_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, fn, block, smem));
    if (b < 1) b = 1;
    ctx->blocks_per_sm[fn] = b;
    *out = b;
    return ACM_OK;
}

int32_t acm_ensure_partials(acm_ctx* ctx, size_t doubles) {
    if (ctx->partials_cap >= doubles) return ACM_OK;
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->d_partials); ctx->d_partials = nullptr; ctx->partials_cap = 0;
    ACM_CUDA(ctx, cudaMalloc(&ctx->d_partials, doubles * sizeof(double)));
    ctx->partials_cap = doubles;
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// point buffers
// ---------------------------------------------------------------------------------------
extern "C" int32_t acm_points_create(acm_ctx* ctx, int32_t dim, size_t n, int32_t dtype, acm_points** out) {
    if (!ctx || !out) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    *out = nullptr;
    ACM_REQUIRE(ctx, dim == 2 || dim == 3, "points: dim must be 2 or 3");
    ACM_REQUIRE(ctx, dtype == ACM_F64 || dtype == ACM_F32, "points: dtype must be ACM_F64 or ACM_F32");
    acm_points* p = new (std::nothrow) acm_points();
    if (!p) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "out of host memory");
    size_t es = dtype == ACM_F64 ? 8 : 4;
    p->dim = dim; p->dtype = dtype; p->n = n;
    p->stride_bytes = ((n * es + 255) / 256) * 256;
    if (p->stride_bytes == 0) p->stride_bytes = 256;
    p->base = nullptr;
    const size_t need = p->stride_bytes * (size_t)dim;
    // best fit from the free list: large enough, at most 50 % (+1 MiB) larger
    int best = -1;
    for (int i = 0; i < ACM_FREE_LIST; ++i)
        if (ctx->free_ptr[i] && ctx->free_bytes[i] >= need && ctx->free_bytes[i] <= need + need / 2 + (1u << 20) &&
            (best < 0 || ctx->free_bytes[i] < ctx->free_bytes[best]))
            best = i;
    if (best >= 0) {
        p->base = ctx->free_ptr[best]; p->alloc_bytes = ctx->free_bytes[best];
        ctx->free_ptr[best] = nullptr; ctx->free_bytes[best] = 0;
    } else {
        cudaError_t e = cudaSetDevice(ctx->device);
        if (e != cudaSuccess) { delete p; return acm_fail(ctx, ACM_ERR_CUDA, "cudaSetDevice failed: %s", cudaGetErrorString(e)); }
        int32_t rc = acm_device_malloc(ctx, &p->base, need);
        if (rc) { delete p; return rc; }
        p->alloc_bytes = need;
    }
    *out = p;
    return ACM_OK;
}

// The buffer is idle once the compute stream has drained (uploads on the copy stream complete inside
// the upload call), so it can be handed to the next acm_points_create without further ordering.
extern "C" int32_t acm_points_destroy(acm_ctx* ctx, acm_points* p) {
    if (!p) return ACM_OK;
    if (ctx) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy_stream);
        // keep allocations up to 16 GiB each; a full list evicts its smallest entry
        if (p->base && p->alloc_bytes <= ((size_t)16 << 30)) {
            int slot = -1, smallest = 0;
            for (int i = 0; i < ACM_FREE_LIST; ++i) {
                if (!ctx->free_ptr[i]) { slot = i; break; }
                if (ctx->free_bytes[i] < ctx->free_bytes[smallest]) smallest = i;
            }
            if (slot < 0 && ctx->free_bytes[smallest] < p->alloc_bytes) { cudaFree(ctx->free_ptr[smallest]); slot = smallest; }
            if (slot >= 0) {
                ctx->free_ptr[slot] = p->base; ctx->free_bytes[slot] = p->alloc_bytes;
                delete p;
                return ACM_OK;
            }
        }
    }
    cudaFree(p->base);
    delete p;
    return ACM_OK;
}
extern "C" size_t acm_points_len(const acm_points* p) { return p ? p->n : 0; }
extern "C" int32_t acm_points_dim(const acm_points* p) { return p ? p->dim : 0; }
extern "C" int32_t acm_points_dtype(const acm_points* p) { return p ? p->dtype : -1; }
extern "C" void* acm_points_component(const acm_points* p, int32_t c) {
    if (!p || c < 0 || c >= p->dim) return nullptr;
    return static_cast<char*>(p->base) + (size_t)c * p->stride_bytes;
}

// AoS (xyzxyz...) f64 staging -> SoA components of type T.  A block stages 256 points through
// shared memory so that both the global read and the global writes are fully coalesced.
template <int DIM, typename T>
__global__ void __launch_bounds__(256) aos_to_soa_kernel(const double* __restrict__ aos, T* __restrict__ c0, T* __restrict__ c1,
                                                         T* __restrict__ c2, size_t n) {
    __shared__ double tile[256 * DIM];
    const size_t nblk = (n + 255) / 256;
    for (size_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const size_t base = blk * 256;
        const size_t cnt = (n - base < 256) ? n - base : 256;
        for (size_t j = threadIdx.x; j < cnt * DIM; j += 256) tile[j] = __ldcs(aos + base * DIM + j);
        __syncthreads();
        if (threadIdx.x < cnt) {
            c0[base + threadIdx.x] = (T)tile[threadIdx.x * DIM];
            c1[base + threadIdx.x] = (T)tile[threadIdx.x * DIM + 1];
            if (DIM == 3) c2[base + threadIdx.x] = (T)tile[threadIdx.x * DIM + 2];
        }
        __syncthreads();
    }
}

template <int DIM, typename T>
__global__ void __launch_bounds__(256) soa_to_aos_kernel(const T* __restrict__ c0, const T* __restrict__ c1, const T* __restrict__ c2,
                                                         double* __restrict__ aos, size_t n) {
    __shared__ double tile[256 * DIM];
    const size_t nblk = (n + 255) / 256;
    for (size_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const size_t base = blk * 256;
        const size_t cnt = (n - base < 256) ? n - base : 256;
        if (threadIdx.x < cnt) {
            tile[threadIdx.x * DIM] = (double)c0[base + threadIdx.x];
            tile[threadIdx.x * DIM + 1] = (double)c1[base + threadIdx.x];
            if (DIM == 3) tile[threadIdx.x * DIM + 2] = (double)c2[base + threadIdx.x];
        }
        __syncthreads();
        for (size_t j = threadIdx.x; j < cnt * DIM; j += 256) aos[base * DIM + j] = tile[j];
        __syncthreads();
    }
}

template <typename T>
static void launch_a2s(acm_ctx* ctx, const acm_points* p, const double* d_aos, size_t off, size_t cnt) {
    int grid = grid_for(ctx, cnt, 256, 8);
    T* c0 = comp<T>(p, 0) + off; T* c1 = comp<T>(p, 1) + off; T* c2 = p->dim == 3 ? comp<T>(p, 2) + off : nullptr;
    if (p->dim == 3) aos_to_soa_kernel<3, T><<<grid, 256, 0, ctx->stream>>>(d_aos, c0, c1, c2, cnt);
    else aos_to_soa_kernel<2, T><<<grid, 256, 0, ctx->stream>>>(d_aos, c0, c1, c2, cnt);
}
template <typename T>
static void launch_s2a(acm_ctx* ctx, const acm_points* p, double* d_aos, size_t off, size_t cnt) {
    int grid = grid_for(ctx, cnt, 256, 8);
    const T* c0 = comp<T>(p, 0) + off; const T* c1 = comp<T>(p, 1) + off; const T* c2 = p->dim == 3 ? comp<T>(p, 2) + off : nullptr;
    if (p->dim == 3) soa_to_aos_kernel<3, T><<<grid, 256, 0, ctx->stream>>>(c0, c1, c2, d_aos, cnt);
    else soa_to_aos_kernel<2, T><<<grid, 256, 0, ctx->stream>>>(c0, c1, c2, d_aos, cnt);
}

static const size_t kChunkPoints = (size_t)4 << 20;  // 4 Mi points per staged chunk (96 MiB for xyz)

// Chunked, double-buffered: H2D of chunk k+1 (copy stream) overlaps the AoS->SoA kernel of
// chunk k (compute stream).  Asynchronous w.r.t. the host only when the source is pinned.
int32_t acm_points_upload_any(acm_ctx* ctx, acm_points* p, const double* host_aos, size_t n, size_t dst_offset) {
    ACM_REQUIRE(ctx, p && (host_aos || n == 0), "upload: null argument");
    ACM_REQUIRE(ctx, dst_offset + n <= p->n, "upload: more points than the buffer holds");
    if (n == 0) return ACM_OK;
    const size_t dim = (size_t)p->dim;
    const size_t chunk = n < kChunkPoints ? n : kChunkPoints;
    int32_t rc = acm_ensure_stage(ctx, chunk * 3 * sizeof(double));
    if (rc) return rc;
    // staging buffers may still be read by kernels enqueued earlier on the compute stream
    ACM_CUDA(ctx, cudaEventRecord(ctx->chunk_ev[2], ctx->stream));
    ACM_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->chunk_ev[2], 0));
    size_t done = 0; int k = 0;
    while (done < n) {
        size_t cnt = (n - done < chunk) ? n - done : chunk;
        int b = k & 1;
        if (k >= 2) ACM_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->chunk_ev[2 + b], 0));  // kernel of chunk k-2 done
        ACM_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage[b], host_aos + done * dim, cnt * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->copy_stream));
        ACM_CUDA(ctx, cudaEventRecord(ctx->chunk_ev[b], ctx->copy_stream));
        ACM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->chunk_ev[b], 0));
        if (p->dtype == ACM_F64) launch_a2s<double>(ctx, p, (const double*)ctx->d_stage[b], dst_offset + done, cnt);
        else launch_a2s<float>(ctx, p, (const double*)ctx->d_stage[b], dst_offset + done, cnt);
        ACM_CHECK_LAUNCH(ctx);
        ACM_CUDA(ctx, cudaEventRecord(ctx->chunk_ev[2 + b], ctx->stream));
        done += cnt; ++k;
    }
    return ACM_OK;
}

extern "C" int32_t acm_points_upload_aos_f64(acm_ctx* ctx, acm_points* p, const double* host_aos, size_t n) {
    ACM_ENTER(ctx);
    return acm_points_upload_any(ctx, p, host_aos, n, 0);
}

extern "C" int32_t acm_points_download_aos_f64(acm_ctx* ctx, const acm_points* p, double* host_aos, size_t n) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, p && (host_aos || n == 0), "download: null argument");
    ACM_REQUIRE(ctx, n <= p->n, "download: more points than the buffer holds");
    if (n == 0) return ACM_OK;
    const size_t dim = (size_t)p->dim;
    const size_t chunk = n < kChunkPoints ? n : kChunkPoints;
    int32_t rc = acm_ensure_stage(ctx, chunk * 3 * sizeof(double));
    if (rc) return rc;
    size_t done = 0;
    while (done < n) {  // simple: kernel then copy on the same stream
        size_t cnt = (n - done < chunk) ? n - done : chunk;
        if (p->dtype == ACM_F64) launch_s2a<double>(ctx, p, (double*)ctx->d_stage[0], done, cnt);
        else launch_s2a<float>(ctx, p, (double*)ctx->d_stage[0], done, cnt);
        ACM_CHECK_LAUNCH(ctx);
        ACM_CUDA(ctx, cudaMemcpyAsync(host_aos + done * dim, ctx->d_stage[0], cnt * dim * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        done += cnt;
    }
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// host-buffer project / unproject (what `CameraModel::project` over nalgebra data binds)
// ---------------------------------------------------------------------------------------
static int32_t host_map(acm_ctx* ctx, const acm_camera* cam, const double* in_aos, size_t n, double* out_aos, uint8_t* status, bool is_project) {
    ACM_REQUIRE(ctx, cam && (n == 0 || (in_aos && out_aos)), "host map: null argument");
    if (n == 0) return ACM_OK;
    if (n <= ACM_SMALL_BATCH) {
        // scalar / small-batch calls (the trait's project(&p)): mapped pinned staging owned by the context, ONE kernel that
        // reads and writes host memory directly.  Single-block batches (n <= 128) do not even synchronise the stream: the
        // kernel publishes a sequence number in the staging area when its results are out and the host spins on it.
        // staging layout, in doubles of ACM_SMALL_BATCH points: input [0, 3N), output [3N, 6N) (a ray takes 3), status bytes
        // at 6N, the sequence flag after them
        const size_t in_dim = is_project ? 3 : 2, out_dim = is_project ? 2 : 3;
        const size_t flag_off = (size_t)ACM_SMALL_BATCH * (6 * sizeof(double) + 8);
        if (!ctx->h_small) {
            ACM_CUDA(ctx, cudaHostAlloc(&ctx->h_small, flag_off + 64, cudaHostAllocMapped));
            ACM_CUDA(ctx, cudaHostGetDevicePointer(&ctx->d_small_alias, ctx->h_small, 0));
            memset(ctx->h_small, 0, flag_off + 64);
            ctx->small_cap = ACM_SMALL_BATCH; ctx->small_seq = 0;
        }
        double* h_in = static_cast<double*>(ctx->h_small);
        double* h_out = h_in + 3 * (size_t)ACM_SMALL_BATCH;
        uint8_t* h_st = reinterpret_cast<uint8_t*>(h_in + 6 * (size_t)ACM_SMALL_BATCH);
        volatile unsigned long long* h_flag = reinterpret_cast<volatile unsigned long long*>(static_cast<char*>(ctx->h_small) + flag_off);
        char* d_base = static_cast<char*>(ctx->d_small_alias);
        double* d_in = reinterpret_cast<double*>(d_base);
        memcpy(h_in, in_aos, n * in_dim * sizeof(double));
        const unsigned long long seq = ++ctx->small_seq;
        int32_t rcs = acm_small_map(ctx, cam, d_in, d_in + 3 * (size_t)ACM_SMALL_BATCH, reinterpret_cast<uint8_t*>(d_in + 6 * (size_t)ACM_SMALL_BATCH),
                                    (int)n, is_project, reinterpret_cast<unsigned long long*>(d_base + flag_off), seq);
        if (rcs) return rcs;
        bool done = false;
        if (n <= 128) {
            const auto t0 = std::chrono::steady_clock::now();
            for (unsigned spins = 0; !done; ++spins) {
                if (*h_flag == seq) { done = true; break; }
                if ((spins & 1023u) == 1023u && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(50)) break;  // slow device: fall back
            }
            std::atomic_thread_fence(std::memory_order_acquire);
        }
        if (!done) ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        memcpy(out_aos, h_out, n * out_dim * sizeof(double));
        if (status) memcpy(status, h_st, n);
        return ACM_OK;
    }
    acm_points *in = nullptr, *out = nullptr;
    uint8_t* d_st = nullptr;
    int32_t rc = acm_points_create(ctx, is_project ? 3 : 2, n, ACM_F64, &in);
    if (!rc) rc = acm_points_create(ctx, is_project ? 2 : 3, n, ACM_F64, &out);
    if (!rc) { rc = acm_ensure_scratch(ctx, n); d_st = static_cast<uint8_t*>(ctx->d_scratch); }
    if (!rc) rc = acm_points_upload_aos_f64(ctx, in, in_aos, n);
    if (!rc) rc = is_project ? acm_project(ctx, cam, in, out, d_st) : acm_unproject(ctx, cam, in, out, d_st);
    if (!rc) rc = acm_points_download_aos_f64(ctx, out, out_aos, n);
    if (!rc && status) {
        cudaError_t e = cudaMemcpyAsync(status, d_st, n, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = acm_fail(ctx, ACM_ERR_CUDA, "status download failed: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(ctx->stream);
    acm_points_destroy(ctx, in);
    acm_points_destroy(ctx, out);
    return rc;
}

extern "C" int32_t acm_project_host(acm_ctx* ctx, const acm_camera* cam, const double* xyz_aos, size_t n, double* uv_aos, uint8_t* status) {
    ACM_ENTER(ctx);
    return host_map(ctx, cam, xyz_aos, n, uv_aos, status, true);
}
extern "C" int32_t acm_unproject_host(acm_ctx* ctx, const acm_camera* cam, const double* uv_aos, size_t n, double* xyz_aos, uint8_t* status) {
    ACM_ENTER(ctx);
    return host_map(ctx, cam, uv_aos, n, xyz_aos, status, false);
}

extern "C" int32_t acm_undistort_rgb8_host(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics, const uint8_t* frames_in,
                                           uint8_t* frames_out, size_t n_frames, int32_t interpolation) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && (n_frames == 0 || (frames_in && frames_out)), "undistort_host: null argument");
    if (n_frames == 0) return ACM_OK;
    size_t fb = (size_t)cam->width * cam->height * 3;
    uint8_t *d_in = nullptr, *d_out = nullptr;
    ACM_CUDA(ctx, cudaMalloc(&d_in, fb * n_frames));
    if (cudaMalloc(&d_out, fb * n_frames) != cudaSuccess) { cudaFree(d_in); return acm_fail(ctx, ACM_ERR_CUDA, "cudaMalloc failed"); }
    int32_t rc = ACM_OK;
    cudaError_t e = cudaMemcpyAsync(d_in, frames_in, fb * n_frames, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) rc = acm_fail(ctx, ACM_ERR_CUDA, "H2D failed: %s", cudaGetErrorString(e));
    if (!rc) rc = acm_undistort_rgb8(ctx, cam, target_intrinsics, d_in, d_out, n_frames, interpolation);
    if (!rc) {
        e = cudaMemcpyAsync(frames_out, d_out, fb * n_frames, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = acm_fail(ctx, ACM_ERR_CUDA, "D2H failed: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(ctx->stream);
    cudaFree(d_in); cudaFree(d_out);
    return rc;
}

// ---------------------------------------------------------------------------------------
// NCCL (loaded at run time so that single-GPU use has no NCCL dependency)
// ---------------------------------------------------------------------------------------
struct NcclId { char internal[128]; };
struct NcclApi {
    void* handle;
    int (*GetUniqueId)(void*);
    int (*CommInitRank)(void**, int, /*ncclUniqueId by value*/ NcclId, int);
    int (*CommDestroy)(void*);
    int (*CommInitAll)(void**, int, const int*);
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    const char* (*GetErrorString)(int);
};
static NcclApi g_nccl = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

static int32_t load_nccl(acm_ctx* ctx) {
    if (g_nccl.handle) return ACM_OK;
    const char* names[] = {"libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"};
    void* h = nullptr;
    const char* env = getenv("ACM_NCCL_LIB");
    if (env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
    for (int i = 0; !h && i < 3; ++i) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!h) return acm_fail(ctx, ACM_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    g_nccl.CommInitAll = (int (*)(void**, int, const int*))dlsym(h, "ncclCommInitAll");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllReduce)
        return acm_fail(ctx, ACM_ERR_NCCL, "libnccl is missing a required symbol");
    g_nccl.handle = h;
    return ACM_OK;
}

static const char* nccl_err(int r) { return g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "nccl error"; }

extern "C" int32_t acm_comm_get_unique_id(uint8_t id[128]) {
    if (!id) return ACM_ERR_INVALID_ARG;
    int32_t rc = load_nccl(nullptr);
    if (rc) return rc;
    int r = g_nccl.GetUniqueId(id);
    if (r != 0) return acm_fail(nullptr, ACM_ERR_NCCL, "ncclGetUniqueId: %s", nccl_err(r));
    return ACM_OK;
}

extern "C" int32_t acm_comm_init_rank(acm_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t id[128]) {
    if (!ctx || !id) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_REQUIRE(ctx, n_ranks >= 1 && rank >= 0 && rank < n_ranks, "comm_init_rank: bad rank / size");
    ACM_REQUIRE(ctx, ctx->comm == nullptr, "comm_init_rank: communicator already attached");
    int32_t rc = load_nccl(ctx);
    if (rc) return rc;
    ACM_CUDA(ctx, cudaSetDevice(ctx->device));
    NcclId nid;
    memcpy(nid.internal, id, 128);
    void* comm = nullptr;
    int r = g_nccl.CommInitRank(&comm, n_ranks, nid, rank);
    if (r != 0) return acm_fail(ctx, ACM_ERR_NCCL, "ncclCommInitRank: %s", nccl_err(r));
    ctx->comm = comm; ctx->n_ranks = n_ranks; ctx->rank = rank;
    return ACM_OK;
}

// One communicator per context of a single-process group (acm_comm_init_all).  libnccl missing is not an error here:
// the fused NVLink exchange does not need it; the entry points that do (linear estimation, statistics) say so.
int32_t acm_nccl_init_all(acm_ctx** ctxs, int32_t n) {
    if (load_nccl(nullptr) != ACM_OK || !g_nccl.CommInitAll) return ACM_OK;
    void* comms[ACM_MAX_PEERS];
    int devs[ACM_MAX_PEERS];
    for (int i = 0; i < n; ++i) devs[i] = ctxs[i]->device;
    int r = g_nccl.CommInitAll(comms, n, devs);
    if (r != 0) return acm_fail(ctxs[0], ACM_ERR_NCCL, "ncclCommInitAll: %s", nccl_err(r));
    for (int i = 0; i < n; ++i) { ctxs[i]->comm = comms[i]; ctxs[i]->n_ranks = n; ctxs[i]->rank = i; }
    return ACM_OK;
}

extern "C" int32_t acm_comm_destroy(acm_ctx* ctx) {
    ACM_ENTER(ctx);
    if (ctx->comm && g_nccl.CommDestroy) { cudaStreamSynchronize(ctx->stream); g_nccl.CommDestroy(ctx->comm); }
    ctx->comm = nullptr; ctx->n_ranks = 1; ctx->rank = 0;
    return ACM_OK;
}

extern "C" int32_t acm_comm_size(const acm_ctx* ctx) { return ctx ? ctx->n_ranks : 0; }

// Sum a small f64 vector over all ranks on the compute stream (no-op without a communicator).
int32_t acm_allreduce_sum_f64(acm_ctx* ctx, double* d_buf, size_t count) {
    if (ctx->n_ranks == 1) return ACM_OK;
    if (!ctx->comm) return acm_fail(ctx, ACM_ERR_NCCL, "this operation needs an NCCL communicator (acm_comm_init_rank) when ranks > 1");
    int r = g_nccl.AllReduce(d_buf, d_buf, count, /*ncclFloat64*/ 8, /*ncclSum*/ 0, ctx->comm, ctx->stream);
    if (r != 0) return acm_fail(ctx, ACM_ERR_NCCL, "ncclAllReduce: %s", nccl_err(r));
    return ACM_OK;
}

int32_t acm_allreduce_sum_u64(acm_ctx* ctx, unsigned long long* d_buf, size_t count) {
    if (ctx->n_ranks == 1) return ACM_OK;
    if (!ctx->comm) return acm_fail(ctx, ACM_ERR_NCCL, "this operation needs an NCCL communicator (acm_comm_init_rank) when ranks > 1");
    int r = g_nccl.AllReduce(d_buf, d_buf, count, /*ncclUint64*/ 5, /*ncclSum*/ 0, ctx->comm, ctx->stream);
    if (r != 0) return acm_fail(ctx, ACM_ERR_NCCL, "ncclAllReduce: %s", nccl_err(r));
    return ACM_OK;
}

// byte-wise maximum (the OR of 0 / 255 image planes drawn by different ranks)
int32_t acm_allreduce_max_u8(acm_ctx* ctx, uint8_t* d_buf, size_t count) {
    if (ctx->n_ranks == 1) return ACM_OK;
    if (!ctx->comm) return acm_fail(ctx, ACM_ERR_NCCL, "this operation needs an NCCL communicator (acm_comm_init_rank) when ranks > 1");
    int r = g_nccl.AllReduce(d_buf, d_buf, count, /*ncclUint8*/ 1, /*ncclMax*/ 2, ctx->comm, ctx->stream);
    if (r != 0) return acm_fail(ctx, ACM_ERR_NCCL, "ncclAllReduce: %s", nccl_err(r));
    return ACM_OK;
}

// Bring the first `count` doubles of ctx->d_reduce of every rank to every host: afterwards
// ctx->h_reduce holds [n_ranks][count] in rank order (stream synchronised).  Every rank writes its
// vector into its own slot of a zero-padded buffer, so the all-reduce acts as an all-gather and
// the caller can combine the slots in rank order -- identical bits on every rank.
int32_t acm_rank_gather_to_host(acm_ctx* ctx, int count) {
    const int R = ctx->n_ranks;
    if (R > 1) {
        if ((size_t)R * count > 1024) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "too many ranks for the gather buffer");
        ACM_CUDA(ctx, cudaMemcpyAsync(ctx->d_partials, ctx->d_reduce, count * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        ACM_CUDA(ctx, cudaMemsetAsync(ctx->d_reduce, 0, (size_t)R * count * sizeof(double), ctx->stream));
        ACM_CUDA(ctx, cudaMemcpyAsync(ctx->d_reduce + (size_t)ctx->rank * count, ctx->d_partials, count * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        int32_t rc = acm_allreduce_sum_f64(ctx, ctx->d_reduce, (size_t)R * count);
        if (rc) return rc;
    }
    ACM_CUDA(ctx, cudaMemcpyAsync(ctx->h_reduce, ctx->d_reduce, (size_t)R * count * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// NVLink peer exchange buffers (CUDA IPC for one process per GPU; direct peer mappings in-process)
// ---------------------------------------------------------------------------------------
static int32_t peer_alloc_local(acm_ctx* ctx) {
    if (ctx->peer_local) return ACM_OK;
    ACM_CUDA(ctx, cudaMalloc(&ctx->peer_local, ACM_PEER_BUFFER_BYTES));
    ACM_CUDA(ctx, cudaMemset(ctx->peer_local, 0, ACM_PEER_BUFFER_BYTES));
    ACM_CUDA(ctx, cudaDeviceSynchronize());
    return ACM_OK;
}

extern "C" int32_t acm_peer_export(acm_ctx* ctx, uint8_t handle[64]) {
    if (!ctx || !handle) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle is 64 bytes");
    int32_t rc = peer_alloc_local(ctx);
    if (rc) return rc;
    cudaIpcMemHandle_t h;
    ACM_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->peer_local));
    memcpy(handle, &h, 64);
    return ACM_OK;
}

// Shared by the IPC form and the in-process form: ptrs[r] = rank r's exchange buffer as seen from this device.
// Every (re-)attach starts from a clean slate: zeroed cells, exchange counter 0, abort flag down.  All ranks must
// have finished their previous exchanges (the caller's barrier) before any of them attaches again.
int32_t acm_peer_setup_pointers(acm_ctx* ctx, int32_t n_ranks, int32_t rank, unsigned char* const* ptrs) {
    ACM_CUDA(ctx, cudaMalloc(&ctx->d_peer_ptrs, ACM_MAX_PEERS * sizeof(unsigned char*)));
    ACM_CUDA(ctx, cudaMemcpy(ctx->d_peer_ptrs, ptrs, n_ranks * sizeof(unsigned char*), cudaMemcpyHostToDevice));
    ctx->peer_n = n_ranks; ctx->peer_rank = rank; ctx->peer_seq = 0; ctx->peer_failed = false;
    if (ctx->n_ranks == 1) { ctx->n_ranks = n_ranks; ctx->rank = rank; }
    return ACM_OK;
}

extern "C" int32_t acm_peer_attach(acm_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t* handles) {
    if (!ctx || !handles) return ACM_ERR_INVALID_ARG;
    acm_bind(ctx);
    ACM_REQUIRE(ctx, n_ranks >= 1 && n_ranks <= ACM_MAX_PEERS && rank >= 0 && rank < n_ranks, "peer_attach: bad rank / size (at most 8 ranks)");
    ACM_REQUIRE(ctx, ctx->peer_local != nullptr, "peer_attach: call acm_peer_export first");
    ACM_REQUIRE(ctx, ctx->peer_n == 0, "peer_attach: peers already attached");
    unsigned char* ptrs[ACM_MAX_PEERS];
    for (int r = 0; r < n_ranks; ++r) {
        if (r == rank) { ptrs[r] = ctx->peer_local; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * 64, 64);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q) if (ctx->peer_mapped[q]) { cudaIpcCloseMemHandle(ctx->peer_mapped[q]); ctx->peer_mapped[q] = nullptr; }
            return acm_fail(ctx, ACM_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
        }
        ctx->peer_mapped[r] = p;
        ptrs[r] = static_cast<unsigned char*>(p);
    }
    return acm_peer_setup_pointers(ctx, n_ranks, rank, ptrs);
}

extern "C" int32_t acm_peer_detach(acm_ctx* ctx) {
    ACM_ENTER(ctx);
    if (ctx->peer_n == 0) return ACM_OK;
    cudaStreamSynchronize(ctx->stream);
    for (int r = 0; r < ACM_MAX_PEERS; ++r) if (ctx->peer_mapped[r]) { cudaIpcCloseMemHandle(ctx->peer_mapped[r]); ctx->peer_mapped[r] = nullptr; }
    cudaFree(ctx->d_peer_ptrs); ctx->d_peer_ptrs = nullptr;
    // the buffer itself stays (its IPC handle may be exported again); wipe it so that a re-attach starts clean
    if (ctx->peer_local) { cudaMemset(ctx->peer_local, 0, ACM_PEER_BUFFER_BYTES); cudaDeviceSynchronize(); }
    ctx->peer_n = 0; ctx->peer_seq = 0; ctx->peer_failed = false;
    if (!ctx->comm) { ctx->n_ranks = 1; ctx->rank = 0; }
    return ACM_OK;
}
