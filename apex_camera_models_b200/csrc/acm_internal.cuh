// Internal declarations shared by the translation units of libacm.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <unordered_map>

#include "../../include/acm.h"

// ---------------------------------------------------------------------------------------
// Camera parameter block passed by value to every kernel (<= 160 B, lives in the kernel's
// constant bank).  k0..k2 are per-model constants the reference recomputes per point; they
// are evaluated once on the host with the reference's own operation order (and glibc's
// tan for FOV) so hoisting them does not change a single bit.
// ---------------------------------------------------------------------------------------
struct CamParams {
    double fx, fy, cx, cy;
    double d[5];
    double W, H;     // resolution as f64 (`width as f64`)
    double k0, k1, k2;
    double ifx, ify;  // RN(1/fx), RN(1/fy) from the host's IEEE division: (u - cx) / fx on the device is then acm_div_by()
    int32_t model;
    int32_t has_resolution;  // width > 0 && height > 0 (kannala_brandt.rs:447-448)
    int32_t fast_div;        // 2^-100 <= |fx|, |fy| <= 2^100: acm_div_by() is bit-identical to the division
    int32_t fast_newton;     // Kannala-Brandt / RadTan: the host-side gate allows the contracted Newton iteration of unproject (acm_make_cam_params)
};

struct acm_points {
    int32_t dim;
    int32_t dtype;
    size_t n;
    size_t stride_bytes;  // distance between components, multiple of 256
    void* base;
    size_t alloc_bytes;   // size of the allocation behind `base` (>= dim * stride_bytes)
};

#define ACM_FREE_LIST 8

// "flag-in-data" cell: a double split over two 8-byte words that each carry half of a 64-bit tag (acm_solver.cu)
struct __align__(16) LLCell { unsigned long long w0, w1; };

#define ACM_MAX_PEERS 8

struct NcclApi;  // dlopen'ed NCCL entry points (acm_core.cu)

struct acm_ctx {
    int device;
    cudaStream_t stream;
    bool owns_stream;
    cudaStream_t copy_stream;  // second stream for chunked host pipelines
    cudaEvent_t t0, t1;
    cudaEvent_t chunk_ev[4];
    int sm_count;
    size_t l2_bytes;
    int cc;
    uint64_t launches;
    std::string err;
    // scratch owned by the context
    double* d_partials;     // per-block partial sums of the reduction kernels
    size_t partials_cap;    // in doubles
    double* d_reduce;       // final reduced vector (2048 doubles; gathers use the first 1024)
    unsigned int* d_ticket; // last-block-done counters
    double* h_reduce;       // pinned mirror of d_reduce (2048 doubles)
    void* d_lm;             // LmState
    void* h_lm;             // pinned mirror
    void* d_stage[2];       // staging for host pipelines
    size_t stage_cap;
    void* h_stage;          // pinned staging for pageable host buffers
    size_t h_stage_cap;
    void* d_scratch;        // grow-only arena for the temporaries of the util entry points
    size_t scratch_cap;
    // destroyed point buffers are kept for the next acm_points_create of a similar size (a
    // cudaMalloc / cudaFree pair costs milliseconds at 10 M points, the kernels around it microseconds)
    void* free_ptr[ACM_FREE_LIST];
    size_t free_bytes[ACM_FREE_LIST];
    acm_points* cache3;     // device buffers kept between *_host calls (grow-only)
    acm_points* cache2;
    size_t cache_cap;
    // NCCL
    void* comm;
    int n_ranks, rank;
    // NVLink peer exchange (acm_peer_*)
    unsigned char* peer_local;   // this rank's exchange buffer (exported through CUDA IPC, or peer-mapped in-process)
    void* peer_mapped[ACM_MAX_PEERS];  // peers' buffers opened in this process through CUDA IPC (nullptr for self / in-process peers)
    unsigned char** d_peer_ptrs; // device array [n_peers] of every rank's buffer, indexed by rank
    int peer_n, peer_rank;
    unsigned long long peer_seq; // exchanges executed so far; advances by the executed count only, identically on every rank
    bool peer_failed;            // an exchange timed out: the ranks are out of step until the peers are re-attached
    struct acm_group* group;     // single-process multi-GPU group this context belongs to (acm_comm_init_all), or nullptr
    unsigned long long lm_tag;   // hand-off tags already handed to lin_kernel launches (never reused)
    LLCell* d_lm_ll;             // flag-in-data hand-off buffers of lin_kernel (block partials + broadcast)
    size_t lm_ll_cap;            // in cells
    int coop_launch;             // cudaDevAttrCooperativeLaunch
    // per-device launch configuration of kernels that need an opt-in (dynamic shared memory above 48 KB) or an occupancy
    // query: attributes and occupancy are per device, so they are cached per context, keyed by the kernel's address
    std::unordered_map<const void*, int> blocks_per_sm;
    // small-batch host path (acm_project_host / acm_unproject_host with few points): mapped pinned staging, no allocation per call
    void* h_small; void* d_small_alias; size_t small_cap; unsigned long long small_seq;
    // the two camera blocks acm_make_cam_params prepared last and their device forms, most recent first (the Newton gates are
    // not free, and a call on a camera pair -- acm_triangulate -- prepares two blocks)
    struct CamCacheEntry { acm_camera key; CamParams val; bool valid; } cam_cache[2];
};

// Make the context's device current on the calling thread (contexts of several GPUs may be driven by one thread).
static inline void acm_bind(const acm_ctx* ctx) {
    int d = -1;
    if (cudaGetDevice(&d) != cudaSuccess || d != ctx->device) cudaSetDevice(ctx->device);
}
#define ACM_ENTER(ctx)                                  \
    do {                                                \
        if (!(ctx)) return ACM_ERR_INVALID_ARG;         \
        acm_bind(ctx);                                  \
    } while (0)

// exchange buffer: 256-byte header (word 0 = sticky abort flag) + 2 alternating sets x ACM_MAX_PEERS rank slots x 64 cells
#define ACM_PEER_HEADER_BYTES 256
#define ACM_PEER_SLOT_CELLS 64
#define ACM_PEER_BUFFER_BYTES (ACM_PEER_HEADER_BYTES + 2 * ACM_MAX_PEERS * ACM_PEER_SLOT_CELLS * sizeof(LLCell))

struct PeerArgs {
    unsigned char* const* bufs;  // nullptr: exchange disabled
    int n_ranks, rank;
    unsigned long long seq;      // number of the (first) exchange this launch executes
};

int32_t acm_fail(acm_ctx* ctx, int32_t code, const char* fmt, ...);
void acm_set_global_error(const char* msg);

#define ACM_CUDA(ctx, call)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess)                                                                \
            return acm_fail((ctx), ACM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define ACM_CHECK_LAUNCH(ctx)                                                                 \
    do {                                                                                      \
        (ctx)->launches++;                                                                    \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess)                                                                \
            return acm_fail((ctx), ACM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define ACM_REQUIRE(ctx, cond, msg)                                                           \
    do {                                                                                      \
        if (!(cond)) return acm_fail((ctx), ACM_ERR_INVALID_ARG, "%s", (msg));                \
    } while (0)

// host helpers implemented in acm_core.cu
int32_t acm_make_cam_params(acm_ctx* ctx, const acm_camera* cam, CamParams* out);
// R (row-major 3x3) must be a proper rotation: finite entries, max |R R^T - I| <= 1e-9, det R > 0.  ctx may be null.
int32_t acm_check_rotation(acm_ctx* ctx, const double* R, const char* who);
int32_t acm_device_malloc(acm_ctx* ctx, void** out, size_t bytes);  // cudaMalloc; empties the free list and retries when out of memory
int32_t acm_ensure_stage(acm_ctx* ctx, size_t bytes);
int32_t acm_ensure_host_stage(acm_ctx* ctx, size_t bytes);
int32_t acm_ensure_partials(acm_ctx* ctx, size_t doubles);
int32_t acm_ensure_scratch(acm_ctx* ctx, size_t bytes);
// resident blocks per SM of a kernel on this context's device (cached); opts in to `smem` bytes of dynamic shared memory above 48 KB
int32_t acm_kernel_blocks_per_sm(acm_ctx* ctx, const void* fn, int block, size_t smem, int* out);
void acm_group_dissolve(acm_ctx* member);
int32_t acm_peer_setup_pointers(acm_ctx* ctx, int32_t n_ranks, int32_t rank, unsigned char* const* ptrs);  // ctx->d_scratch holds >= bytes afterwards (256-byte aligned)
int32_t acm_allreduce_sum_f64(acm_ctx* ctx, double* d_buf, size_t count);
int32_t acm_allreduce_sum_u64(acm_ctx* ctx, unsigned long long* d_buf, size_t count);
int32_t acm_allreduce_max_u8(acm_ctx* ctx, uint8_t* d_buf, size_t count);
int32_t acm_rank_gather_to_host(acm_ctx* ctx, int count);  // d_reduce[0..count) of every rank -> h_reduce[rank][count]
// project / unproject of n <= ACM_SMALL_BATCH AoS points that sit in device-visible (mapped pinned) memory (acm_exact.cu)
#define ACM_SMALL_BATCH 2048
int32_t acm_small_map(acm_ctx* ctx, const acm_camera* cam, const double* d_in, double* d_out, uint8_t* d_status, int n, bool is_project,
                      unsigned long long* d_done_flag, unsigned long long seq);
int32_t acm_points_upload_any(acm_ctx* ctx, acm_points* p, const double* host_aos, size_t n, size_t dst_offset);

template <typename T>
static inline T* comp(const acm_points* p, int c) {
    return reinterpret_cast<T*>(static_cast<char*>(p->base) + (size_t)c * p->stride_bytes);
}

static inline int grid_for(const acm_ctx* ctx, size_t work_items, int block, int blocks_per_sm) {
    size_t need = (work_items + (size_t)block - 1) / (size_t)block;
    size_t cap = (size_t)ctx->sm_count * (size_t)blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}
