// acm.hpp -- C++ host layer above the C ABI (include/acm.h).
//
// The reference is compiled Rust and its toolchain is absent here, so this header is the native
// host-side mirror of its interface for the hot path: the `CameraModel` trait (reference
// src/camera/mod.rs:241-340: project, unproject, load_from_yaml, save_to_yaml, validate_params,
// get_resolution, get_intrinsics, get_distortion, get_model_name), each model's `new(&DVector)` and
// `linear_estimation`, the README-era `*OptimizationCost` (README.md:70-81) and the util hot loops.
// Header-only; link with -lacm.  Errors are the reference's `CameraModelError` variants.
#pragma once
#include <array>
#include <cmath>
#include <cstdint>
#include <fstream>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "acm.h"

namespace acm {

struct Intrinsics { double fx, fy, cx, cy; };   // mod.rs:52-62
struct Resolution { uint32_t width, height; };  // mod.rs:67-73
using Vector2 = std::array<double, 2>;
using Vector3 = std::array<double, 3>;

enum class ErrorKind {  // mod.rs:79-113 (+ Library for CUDA/NCCL failures)
    ProjectionOutSideImage, PointIsOutSideImage, PointAtCameraCenter, FocalLengthMustBePositive,
    PrincipalPointMustBeFinite, InvalidParams, YamlError, IOError, NumericalError, ZeroProjectionPoints, Library
};

class CameraModelError : public std::runtime_error {
public:
    ErrorKind kind;
    CameraModelError(ErrorKind k, const std::string& msg) : std::runtime_error(msg), kind(k) {}
};

inline void throw_point_status(uint8_t st, int model) {
    switch (st) {
        case ACM_POINT_OK: return;
        case ACM_POINT_IS_OUTSIDE_IMAGE: throw CameraModelError(ErrorKind::PointIsOutSideImage, "Input point is outside the image");
        case ACM_POINT_AT_CAMERA_CENTER: throw CameraModelError(ErrorKind::PointAtCameraCenter, "z is close to zero, point is at camera center");
        case ACM_PROJECTION_OUTSIDE_IMAGE: throw CameraModelError(ErrorKind::ProjectionOutSideImage, "Projection is outside the image");
        default: throw CameraModelError(ErrorKind::NumericalError, model == ACM_MODEL_RADTAN ? "NumericalError: Jacobian is singular" : "NumericalError: Unprojection failed to converge");
    }
}

inline void throw_call_status(int32_t rc, const std::string& msg) {
    switch (rc) {
        case ACM_OK: return;
        case ACM_ERR_INVALID_PARAMS: throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: " + msg);
        case ACM_ERR_NUMERICAL: throw CameraModelError(ErrorKind::NumericalError, "NumericalError: " + msg);
        case ACM_ERR_FOCAL_LENGTH: throw CameraModelError(ErrorKind::FocalLengthMustBePositive, "Focal length must be positive");
        case ACM_ERR_PRINCIPAL_POINT: throw CameraModelError(ErrorKind::PrincipalPointMustBeFinite, "Principal point must be finite");
        case ACM_ERR_ZERO_PROJECTION_POINTS: throw CameraModelError(ErrorKind::ZeroProjectionPoints, "Zero projection points");
        default: throw CameraModelError(ErrorKind::Library, "libacm error " + std::to_string(rc) + ": " + msg);
    }
}

class Context {
public:
    explicit Context(int device = 0, void* stream = nullptr) {
        int32_t rc = acm_ctx_create(device, stream, &h_);
        if (rc != ACM_OK) throw CameraModelError(ErrorKind::Library, std::string("acm_ctx_create: ") + acm_last_error(nullptr));
    }
    ~Context() { if (h_) acm_ctx_destroy(h_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    acm_ctx* handle() const { return h_; }
    void check(int32_t rc) const { if (rc != ACM_OK) throw_call_status(rc, acm_last_error(h_)); }
    void sync() const { check(acm_ctx_sync(h_)); }
private:
    acm_ctx* h_ = nullptr;
};

// Device SoA buffer; host memory order is nalgebra's (xyzxyz.. / uvuv..).
class Points {
public:
    Points(const Context& ctx, int dim, size_t n, int dtype = ACM_F64) : ctx_(&ctx) { ctx.check(acm_points_create(ctx.handle(), dim, n, dtype, &h_)); }
    Points(const Context& ctx, int dim, const double* host_aos, size_t n) : Points(ctx, dim, n) { upload(host_aos, n); }
    Points(const Context& ctx, acm_points* adopt) : ctx_(&ctx), h_(adopt) {}
    ~Points() { if (h_) acm_points_destroy(ctx_->handle(), h_); }
    Points(const Points&) = delete;
    Points& operator=(const Points&) = delete;
    Points(Points&& o) noexcept : ctx_(o.ctx_), h_(o.h_) { o.h_ = nullptr; }
    void upload(const double* host_aos, size_t n) { ctx_->check(acm_points_upload_aos_f64(ctx_->handle(), h_, host_aos, n)); ctx_->sync(); }
    std::vector<double> download() const {
        std::vector<double> out(size() * (size_t)acm_points_dim(h_));
        ctx_->check(acm_points_download_aos_f64(ctx_->handle(), h_, out.data(), size()));
        return out;
    }
    size_t size() const { return acm_points_len(h_); }
    acm_points* handle() const { return h_; }
private:
    const Context* ctx_;
    acm_points* h_ = nullptr;
};

namespace detail {
// Minimal reader for the calibration YAML the reference uses (samples/*.yaml): `cam0:` mapping with
// flow sequences of numbers (possibly spread over several lines) under named keys.
inline bool find_sequence(const std::string& text, const std::string& key, std::vector<double>& out, bool& all_int, bool& all_float) {
    size_t pos = text.find("\n  " + key + ":");
    if (pos == std::string::npos) pos = text.find(" " + key + ":");
    if (pos == std::string::npos) return false;
    size_t lb = text.find('[', pos), rb = text.find(']', pos);
    if (lb == std::string::npos || rb == std::string::npos || rb < lb) return false;
    std::string body = text.substr(lb + 1, rb - lb - 1);
    for (char& c : body) if (c == ',' || c == '\n' || c == '\r' || c == '\t') c = ' ';
    std::istringstream is(body);
    std::string tok;
    out.clear(); all_int = true; all_float = true;
    while (is >> tok) {
        try { size_t used = 0; double v = std::stod(tok, &used); if (used != tok.size()) return false; out.push_back(v); }
        catch (...) { return false; }
        bool is_float = tok.find_first_of(".eEnN") != std::string::npos;
        all_int = all_int && !is_float; all_float = all_float && is_float;
    }
    return true;
}
}  // namespace detail

class CameraModel {
public:
    Intrinsics intrinsics{0, 0, 0, 0};
    Resolution resolution{0, 0};
    std::vector<double> distortions;

    virtual ~CameraModel() = default;
    virtual int model_id() const = 0;
    virtual const char* get_model_name() const = 0;
    virtual const char* yaml_distortion_key() const { return nullptr; }       // KB / RadTan keep distortion outside `intrinsics`
    virtual const char* yaml_save_distortion_key() const { return yaml_distortion_key(); }

    void bind(const Context& ctx) { ctx_ = &ctx; }
    const Context& ctx() const { if (!ctx_) throw CameraModelError(ErrorKind::Library, "camera model is not bound to a Context"); return *ctx_; }

    acm_camera block() const {
        acm_camera c{};
        c.model = model_id(); c.width = resolution.width; c.height = resolution.height;
        c.n_params = (int32_t)(4 + distortions.size());
        c.params[0] = intrinsics.fx; c.params[1] = intrinsics.fy; c.params[2] = intrinsics.cx; c.params[3] = intrinsics.cy;
        for (size_t i = 0; i < distortions.size(); ++i) c.params[4 + i] = distortions[i];
        return c;
    }
    void set_params(const double* p, size_t n) {
        intrinsics = {p[0], p[1], p[2], p[3]};
        distortions.assign(p + 4, p + n);
    }

    // ---- trait ---------------------------------------------------------------------------
    Vector2 project(const Vector3& p) const {
        Vector2 uv; uint8_t st;
        project_batch(p.data(), 1, uv.data(), &st);
        throw_point_status(st, model_id());
        return uv;
    }
    Vector3 unproject(const Vector2& p) const {
        Vector3 ray; uint8_t st;
        unproject_batch(p.data(), 1, ray.data(), &st);
        throw_point_status(st, model_id());
        return ray;
    }
    void project_batch(const double* xyz_aos, size_t n, double* uv_aos, uint8_t* status) const {
        acm_camera c = block();
        ctx().check(acm_project_host(ctx().handle(), &c, xyz_aos, n, uv_aos, status));
    }
    void unproject_batch(const double* uv_aos, size_t n, double* xyz_aos, uint8_t* status) const {
        acm_camera c = block();
        ctx().check(acm_unproject_host(ctx().handle(), &c, uv_aos, n, xyz_aos, status));
    }
    void validate_params() const {
        char msg[256] = "";
        acm_camera c = block();
        throw_call_status(acm_validate_params(&c, msg, sizeof(msg)), msg);
    }
    Resolution get_resolution() const { return resolution; }
    Intrinsics get_intrinsics() const { return intrinsics; }
    std::vector<double> get_distortion() const { return distortions; }

    // inherent linear_estimation(&mut self, &Matrix3xX, &Matrix2xX)
    void linear_estimation(const Points& points_3d, const Points& points_2d) {
        acm_camera c = block();
        ctx().check(acm_linear_estimation(ctx().handle(), &c, points_3d.handle(), points_2d.handle()));
        set_params(c.params, (size_t)c.n_params);
    }

    void save_to_yaml(const std::string& path) const {
        std::ofstream f(path);
        if (!f) throw CameraModelError(ErrorKind::IOError, "IO Error: cannot create " + path);
        f.precision(17);
        f << "cam0:\n  camera_model: " << get_model_name() << "\n  intrinsics: [" << intrinsics.fx << ", " << intrinsics.fy << ", " << intrinsics.cx << ", " << intrinsics.cy;
        const char* key = yaml_save_distortion_key();
        auto as_float = [](double v) { std::ostringstream s; s.precision(17); s << v; std::string t = s.str(); if (t.find_first_of(".eEn") == std::string::npos) t += ".0"; return t; };
        if (!key) for (double d : distortions) f << ", " << as_float(d);
        f << "]\n";
        if (key) { f << "  " << key << ": ["; for (size_t i = 0; i < distortions.size(); ++i) f << (i ? ", " : "") << as_float(distortions[i]); f << "]\n"; }
        f << "  resolution: [" << resolution.width << ", " << resolution.height << "]\n";
    }

protected:
    // shared by the derived load_from_yaml (mod.rs:412-501 + per-model distortion handling)
    void load_yaml_into(const std::string& path, size_t n_dist) {
        std::ifstream f(path);
        if (!f) throw CameraModelError(ErrorKind::IOError, "IO Error: cannot read " + path);
        std::stringstream ss; ss << f.rdbuf();
        std::string text = "\n" + ss.str();
        if (text.find("cam0:") == std::string::npos) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: Missing 'cam0' node in YAML");
        std::vector<double> intr, res, dist; bool ai, af;
        if (!detail::find_sequence(text, "intrinsics", intr, ai, af)) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: YAML missing 'intrinsics' array under 'cam0'");
        const char* key = yaml_distortion_key();
        size_t need = key ? 4 : 4 + n_dist;
        if (intr.size() < need) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: Intrinsics array must have at least " + std::to_string(need) + " elements, got " + std::to_string(intr.size()));
        if (!detail::find_sequence(text, "resolution", res, ai, af)) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: YAML missing 'resolution' array under 'cam0'");
        if (res.size() < 2) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: Resolution array must have at least 2 elements (width, height)");
        if (!ai) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: Invalid width: not an integer");
        if (key) {
            if (!detail::find_sequence(text, key, dist, ai, af) || dist.size() < n_dist) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: Missing distortion parameters");
            dist.resize(n_dist);
        } else {
            dist.assign(intr.begin() + 4, intr.end());
            if (dist.size() != n_dist) throw CameraModelError(ErrorKind::InvalidParams, "Invalid camera parameters: expected exactly " + std::to_string(4 + n_dist) + " parameters, got " + std::to_string(intr.size()));
        }
        intrinsics = {intr[0], intr[1], intr[2], intr[3]};
        resolution = {(uint32_t)res[0], (uint32_t)res[1]};
        distortions = dist;
        validate_params();
    }
    void init_from_params(const std::vector<double>& p) {
        acm_camera c{}; char msg[256] = "";
        throw_call_status(acm_camera_new(model_id(), p.data(), p.size(), &c, msg, sizeof(msg)), msg);
        set_params(c.params, (size_t)c.n_params);
        resolution = {0, 0};
    }
private:
    const Context* ctx_ = nullptr;
};

#define ACM_DEFINE_MODEL(Class, Id, Name, NDist, LoadKey, SaveKey)                                        \
    class Class : public CameraModel {                                                                    \
    public:                                                                                               \
        int model_id() const override { return Id; }                                                      \
        const char* get_model_name() const override { return Name; }                                      \
        const char* yaml_distortion_key() const override { return LoadKey; }                              \
        const char* yaml_save_distortion_key() const override { return SaveKey; }                         \
        /* `Class::new(&DVector<f64>)` */                                                                 \
        static Class create(const std::vector<double>& parameters) { Class m; m.init_from_params(parameters); return m; } \
        static Class load_from_yaml(const std::string& path) { Class m; m.load_yaml_into(path, NDist); return m; }       \
    };

ACM_DEFINE_MODEL(PinholeModel, ACM_MODEL_PINHOLE, "pinhole", 0, nullptr, nullptr)
ACM_DEFINE_MODEL(RadTanModel, ACM_MODEL_RADTAN, "rad_tan", 5, "distortion", "distortion")
ACM_DEFINE_MODEL(KannalaBrandtModel, ACM_MODEL_KANNALA_BRANDT, "kannala_brandt", 4, "distortion", "distortion_coeffs")  // kannala_brandt.rs:635 vs :737
ACM_DEFINE_MODEL(UcmModel, ACM_MODEL_UCM, "ucm", 1, nullptr, nullptr)
ACM_DEFINE_MODEL(EucmModel, ACM_MODEL_EUCM, "eucm", 2, nullptr, nullptr)
ACM_DEFINE_MODEL(DoubleSphereModel, ACM_MODEL_DOUBLE_SPHERE, "double_sphere", 2, nullptr, nullptr)
ACM_DEFINE_MODEL(FovModel, ACM_MODEL_FOV, "fov", 1, nullptr, nullptr)
#undef ACM_DEFINE_MODEL

// README-era `XOptimizationCost::new(model, points_3d, points_2d)` -> linear_estimation() -> optimize()
class OptimizationCost {
public:
    OptimizationCost(CameraModel& model, const double* points_3d_aos, const double* points_2d_aos, size_t n, int residual_kind = -1)
        : model_(model), xyz_(model.ctx(), 3, points_3d_aos, n), uv_(model.ctx(), 2, points_2d_aos, n) {
        const int id = model.model_id();
        const bool unified = id == ACM_MODEL_UCM || id == ACM_MODEL_EUCM || id == ACM_MODEL_DOUBLE_SPHERE;
        kind_ = residual_kind >= 0 ? residual_kind : (unified ? ACM_RESIDUAL_ALGEBRAIC : ACM_RESIDUAL_PIXEL);
    }
    void linear_estimation() { model_.linear_estimation(xyz_, uv_); }
    acm_normal_equations linearize() const {
        acm_camera c = model_.block(); acm_normal_equations ne;
        model_.ctx().check(acm_linearize(model_.ctx().handle(), &c, kind_, xyz_.handle(), uv_.handle(), &ne));
        return ne;
    }
    acm_lm_result optimize(const double* lower = nullptr, const double* upper = nullptr, const acm_lm_config* cfg = nullptr) {
        acm_camera c = model_.block(); double out[ACM_MAX_PARAMS]; acm_lm_result res{};
        model_.ctx().check(acm_lm_solve(model_.ctx().handle(), &c, kind_, xyz_.handle(), uv_.handle(), lower, upper, cfg, out, &res));
        model_.set_params(out, (size_t)c.n_params);
        return res;
    }
    Intrinsics get_intrinsics() const { return model_.get_intrinsics(); }
    std::vector<double> get_distortion() const { return model_.get_distortion(); }
private:
    CameraModel& model_;
    Points xyz_, uv_;
    int kind_;
};

// `project(&p, compute_jacobian = true)` in its 2x3 reading (trait doc mod.rs:246-252): uv (2n, nalgebra order) and the
// point Jacobians as n row-major 2x3 blocks [du/dx du/dy du/dz dv/dx dv/dy dv/dz]; status = geometric validity
inline void project_point_jacobian(const CameraModel& m, const double* xyz_aos, size_t n, std::vector<double>& uv_aos,
                                   std::vector<double>& jac, std::vector<uint8_t>& status) {
    const Context& ctx = m.ctx();
    Points X(ctx, 3, xyz_aos, n), U(ctx, 2, n);
    void *dj = nullptr, *ds = nullptr;
    ctx.check(acm_device_alloc(ctx.handle(), (n ? n : 1) * 6 * sizeof(double), &dj));
    ctx.check(acm_device_alloc(ctx.handle(), n ? n : 1, &ds));
    acm_camera c = m.block();
    int32_t rc = acm_project_point_jacobian(ctx.handle(), &c, X.handle(), U.handle(), static_cast<double*>(dj), static_cast<uint8_t*>(ds));
    std::vector<double> rows(6 * n);
    status.assign(n, 0);
    if (rc == ACM_OK && n) rc = acm_memcpy_d2h(ctx.handle(), rows.data(), dj, 6 * n * sizeof(double));
    if (rc == ACM_OK && n) rc = acm_memcpy_d2h(ctx.handle(), status.data(), ds, n);
    if (rc == ACM_OK) rc = acm_ctx_sync(ctx.handle());
    acm_device_free(ctx.handle(), dj); acm_device_free(ctx.handle(), ds);
    ctx.check(rc);
    uv_aos = U.download();
    jac.resize(6 * n);
    for (size_t i = 0; i < n; ++i) for (int k = 0; k < 6; ++k) jac[6 * i + k] = rows[(size_t)k * n + i];
}

// util::compute_reprojection_error (error_metrics.rs:62-121)
inline acm_projection_error compute_reprojection_error(const CameraModel& m, const double* xyz_aos, const double* uv_aos, size_t n) {
    Points X(m.ctx(), 3, xyz_aos, n), U(m.ctx(), 2, uv_aos, n);
    acm_camera c = m.block(); acm_projection_error out{};
    m.ctx().check(acm_reprojection_error(m.ctx().handle(), &c, X.handle(), U.handle(), &out));
    return out;
}

// util::sample_points (point_sampling.rs:46-120): returns (points_2d, points_3d) in nalgebra memory order
// (shard, n_shards): that contiguous slice of the grid, one per GPU
inline std::pair<std::vector<double>, std::vector<double>> sample_points(const CameraModel& m, size_t n, int shard = 0, int n_shards = 1) {
    acm_camera c = m.block(); acm_points *uv = nullptr, *xyz = nullptr; size_t kept = 0;
    m.ctx().check(acm_sample_points_shard(m.ctx().handle(), &c, n, shard, n_shards, &uv, &xyz, &kept));
    Points U(m.ctx(), uv), X(m.ctx(), xyz);
    return {U.download(), X.download()};
}

// util::undistort_image (undistort.rs:14-49): RGB8 interleaved, w*h*3 bytes; interpolation = ACM_INTERP_*
inline std::vector<uint8_t> undistort_image(const std::vector<uint8_t>& image, uint32_t width, uint32_t height, const CameraModel& m,
                                            const Intrinsics* target = nullptr, int interpolation = ACM_INTERP_BILINEAR) {
    if (width != m.resolution.width || height != m.resolution.height)
        throw CameraModelError(ErrorKind::InvalidParams, "Invalid parameters: Image " + std::to_string(width) + "x" + std::to_string(height) + " doesn't match model " +
                                                             std::to_string(m.resolution.width) + "x" + std::to_string(m.resolution.height));
    std::vector<uint8_t> out(image.size());
    acm_camera c = m.block();
    double t[4]; if (target) { t[0] = target->fx; t[1] = target->fy; t[2] = target->cx; t[3] = target->cy; }
    m.ctx().check(acm_undistort_rgb8_host(m.ctx().handle(), &c, target ? t : nullptr, image.data(), out.data(), 1, interpolation));
    return out;
}

// RGB8 frames of `input`'s camera rendered as `output`'s camera sees them (beyond the reference: output.unproject,
// input.project, interpolate_pixel of undistort.rs:51-105).  output == nullptr: undistort_image of `input` with `target`.
// The source coordinates are computed once on the device (32 bytes per output pixel) and reused by every apply().
class RemapPlan {
public:
    RemapPlan(const CameraModel& input, const CameraModel* output, const Intrinsics* target = nullptr, int interpolation = ACM_INTERP_BILINEAR)
        : ctx_(&input.ctx()), in_(input.resolution), out_(output ? output->resolution : input.resolution) {
        acm_camera ci = input.block(), co{};
        if (output) co = output->block();
        double t[4]; if (target) { t[0] = target->fx; t[1] = target->fy; t[2] = target->cx; t[3] = target->cy; }
        ctx_->check(acm_remap_plan_create(ctx_->handle(), &ci, output ? &co : nullptr, target ? t : nullptr, interpolation, &h_));
    }
    // rotated plan (stereo rectification): R row-major with x_out = R x_in (OpenCV's R1 / R2); ray_in = R^T ray_out
    RemapPlan(const CameraModel& input, const CameraModel& output, const std::array<double, 9>& R, int interpolation = ACM_INTERP_BILINEAR)
        : ctx_(&input.ctx()), in_(input.resolution), out_(output.resolution) {
        const acm_camera ci = input.block(), co = output.block();
        ctx_->check(acm_remap_plan_create_rotated(ctx_->handle(), &ci, &co, R.data(), interpolation, &h_));
    }
    ~RemapPlan() { if (h_) acm_remap_plan_destroy(ctx_->handle(), h_); }
    RemapPlan(const RemapPlan&) = delete;
    RemapPlan& operator=(const RemapPlan&) = delete;
    // whole input frames (w*h*3 bytes each) on the host -> output frames
    std::vector<uint8_t> apply(const std::vector<uint8_t>& frames) const {
        const size_t fin = (size_t)in_.width * in_.height * 3;
        if (frames.size() % fin != 0)
            throw CameraModelError(ErrorKind::InvalidParams, "Invalid parameters: frames of " + std::to_string(frames.size()) +
                                                                 " bytes don't match model " + std::to_string(in_.width) + "x" + std::to_string(in_.height));
        const size_t n = frames.size() / fin;
        std::vector<uint8_t> out(n * out_.width * out_.height * 3);
        ctx_->check(acm_remap_rgb8_host(ctx_->handle(), h_, frames.data(), out.data(), n));
        return out;
    }
    // frames resident on the device, enqueued on the context's stream
    void apply_device(const uint8_t* d_in, uint8_t* d_out, size_t n_frames) const {
        ctx_->check(acm_remap_rgb8(ctx_->handle(), h_, d_in, d_out, n_frames));
    }
    Resolution output_resolution() const { return out_; }
    acm_remap_plan* handle() const { return h_; }
private:
    const Context* ctx_;
    Resolution in_, out_;
    acm_remap_plan* h_ = nullptr;
};

// one RGB8 image of `input`'s camera (w*h*3 bytes) as `output`'s camera sees it
inline std::vector<uint8_t> remap_image(const std::vector<uint8_t>& image, uint32_t width, uint32_t height, const CameraModel& input,
                                        const CameraModel& output, int interpolation = ACM_INTERP_BILINEAR) {
    if (width != input.resolution.width || height != input.resolution.height || image.size() != (size_t)width * height * 3)
        throw CameraModelError(ErrorKind::InvalidParams, "Invalid parameters: Image " + std::to_string(width) + "x" + std::to_string(height) + " doesn't match model " +
                                                             std::to_string(input.resolution.width) + "x" + std::to_string(input.resolution.height));
    return RemapPlan(input, &output, nullptr, interpolation).apply(image);
}

// Bouguet rectification of a calibrated pair, x_cam2 = R x_cam1 + t (the rotation part of OpenCV's stereoRectify; host
// only).  x_rect1 = R1 x_cam1, x_rect2 = R2 x_cam2; baseline = the component of R2 t along x (along y when vertical).
// With one Pinhole camera K for both views, P1 = K [I | 0] and P2 = K [I | baseline e].
struct StereoRectification {
    std::array<double, 9> R1, R2;
    double baseline;
    bool vertical;
};

inline StereoRectification stereo_rectify(const std::array<double, 9>& R, const std::array<double, 3>& t) {
    StereoRectification s{};
    int32_t vertical = 0;
    const int32_t rc = acm_stereo_rectify(R.data(), t.data(), s.R1.data(), s.R2.data(), &s.baseline, &vertical);
    if (rc != ACM_OK) throw_call_status(rc, acm_last_error(nullptr));
    s.vertical = vertical != 0;
    return s;
}

// Triangulation of matched pixels of a calibrated pair, x_cam2 = R x_cam1 + t (acm_triangulate_host): points in the first
// camera's frame (NaN where status != ACM_TRI_OK), per-pair pixel errors in both cameras and the ACM_TRI_* status.
// max_iterations = 0: the midpoint of the rays' closest approach; > 0: at most that many Levenberg-Marquardt trials.
struct Triangulation {
    std::vector<double> points;  // xyz per pair (Matrix3xX memory order)
    std::vector<double> errors;  // |first.project(X) - uv1|, |second.project(R X + t) - uv2| per pair
    std::vector<uint8_t> status;
};

inline Triangulation triangulate(const CameraModel& first, const CameraModel& second, const std::array<double, 9>& R,
                                 const std::array<double, 3>& t, const double* uv1_aos, const double* uv2_aos, size_t n,
                                 int32_t max_iterations = 10) {
    Triangulation out;
    out.points.resize(3 * n); out.errors.resize(2 * n); out.status.resize(n);
    const acm_camera a = first.block(), b = second.block();
    first.ctx().check(acm_triangulate_host(first.ctx().handle(), &a, &b, R.data(), t.data(), uv1_aos, uv2_aos, n, max_iterations,
                                           out.points.data(), out.errors.data(), out.status.data()));
    return out;
}

// Depth images of `cam`'s camera (W x H = its resolution, row-major), x_cam = R x + t (acm_render_depth_host): per pixel the
// f32 range |x_cam| of the nearest drawn point and its index; empty pixels hold range bits 0xFFFFFFFF (a NaN) and index
// UINT32_MAX.  Depth is the range along the ray, not z.
struct DepthImage {
    std::vector<float> range;
    std::vector<uint32_t> index;
};

inline DepthImage render_depth(const CameraModel& cam, const std::array<double, 9>& R, const std::array<double, 3>& t,
                               const double* xyz_aos, size_t n) {
    DepthImage out;
    const size_t npix = (size_t)cam.resolution.width * cam.resolution.height;
    out.range.resize(npix); out.index.resize(npix);
    const acm_camera c = cam.block();
    cam.ctx().check(acm_render_depth_host(cam.ctx().handle(), &c, R.data(), t.data(), xyz_aos, n, out.range.data(), out.index.data()));
    return out;
}

// Back-projection of a W x H range image (acm_depth_to_points): x = R^T (unproject(pixel) * range - t) per pixel (Matrix3xX
// memory order, NaN where status != ACM_DEPTH_OK) and the ACM_DEPTH_* status.
struct DepthPoints {
    std::vector<double> points;
    std::vector<uint8_t> status;
};

inline DepthPoints depth_to_points(const CameraModel& cam, const std::array<double, 9>& R, const std::array<double, 3>& t, const float* range) {
    const Context& ctx = cam.ctx();
    const size_t npix = (size_t)cam.resolution.width * cam.resolution.height;
    void* d = nullptr;  // range, then the status bytes
    ctx.check(acm_device_alloc(ctx.handle(), npix ? 5 * npix : 5, &d));
    DepthPoints out;
    try {
        Points X(ctx, 3, npix);
        ctx.check(acm_memcpy_h2d(ctx.handle(), d, range, 4 * npix));
        const acm_camera c = cam.block();
        uint8_t* d_status = static_cast<uint8_t*>(d) + 4 * npix;
        ctx.check(acm_depth_to_points(ctx.handle(), &c, R.data(), t.data(), static_cast<const float*>(d), X.handle(), d_status));
        out.status.resize(npix);
        ctx.check(acm_memcpy_d2h(ctx.handle(), out.status.data(), d_status, npix));
        out.points = X.download();
        ctx.sync();
    } catch (...) {
        acm_device_free(ctx.handle(), d);
        throw;
    }
    acm_device_free(ctx.handle(), d);
    return out;
}

// ---- util::image_quality (image_quality.rs) on RGB8 interleaved images (w*h*3 bytes) --------------
struct ImageQualityMetrics { double psnr, ssim; };   // image_quality.rs:20-26

// RGB8 image staged in HBM for the duration of a call
class DeviceImage {
public:
    DeviceImage(const Context& ctx, size_t bytes, const uint8_t* host = nullptr) : ctx_(ctx), bytes_(bytes) {
        ctx_.check(acm_device_alloc(ctx_.handle(), bytes ? bytes : 4, &p_));
        if (bytes && host) ctx_.check(acm_memcpy_h2d(ctx_.handle(), p_, host, bytes));
        else if (bytes) ctx_.check(acm_memset_d(ctx_.handle(), p_, 0, bytes));
    }
    ~DeviceImage() { if (p_) acm_device_free(ctx_.handle(), p_); }
    DeviceImage(const DeviceImage&) = delete;
    DeviceImage& operator=(const DeviceImage&) = delete;
    uint8_t* ptr() const { return static_cast<uint8_t*>(p_); }
    std::vector<uint8_t> download() const {
        std::vector<uint8_t> out(bytes_);
        if (bytes_) { ctx_.check(acm_memcpy_d2h(ctx_.handle(), out.data(), p_, bytes_)); ctx_.check(acm_ctx_sync(ctx_.handle())); }
        return out;
    }
private:
    const Context& ctx_; size_t bytes_; void* p_ = nullptr;
};

inline void require_same_size(const std::vector<uint8_t>& a, const std::vector<uint8_t>& b, uint32_t w, uint32_t h) {
    if (a.size() != b.size() || a.size() != (size_t)w * h * 3)   // image_quality.rs:46-50, :109-113
        throw CameraModelError(ErrorKind::InvalidParams, "Invalid parameters: Images must have the same dimensions");
}
// util::calculate_psnr (image_quality.rs:45-89)
inline double calculate_psnr(const Context& ctx, const std::vector<uint8_t>& img1, const std::vector<uint8_t>& img2, uint32_t w, uint32_t h) {
    require_same_size(img1, img2, w, h);
    DeviceImage a(ctx, img1.size(), img1.data()), b(ctx, img2.size(), img2.data());
    double out = 0.0;
    ctx.check(acm_image_psnr(ctx.handle(), a.ptr(), b.ptr(), w, h, &out));
    return out;
}
// util::calculate_ssim (image_quality.rs:108-210)
inline double calculate_ssim(const Context& ctx, const std::vector<uint8_t>& img1, const std::vector<uint8_t>& img2, uint32_t w, uint32_t h) {
    require_same_size(img1, img2, w, h);
    DeviceImage a(ctx, img1.size(), img1.data()), b(ctx, img2.size(), img2.data());
    double out = 0.0;
    ctx.check(acm_image_ssim(ctx.handle(), a.ptr(), b.ptr(), w, h, &out));
    return out;
}
// create_projection_image (image_quality.rs:338-373) with one colour: radius-2 discs on black
inline std::vector<uint8_t> create_projection_image(const Context& ctx, const double* uv_aos, size_t n, uint8_t r, uint8_t g, uint8_t b, uint32_t w, uint32_t h) {
    DeviceImage img(ctx, (size_t)w * h * 3);
    Points U(ctx, 2, uv_aos, n);
    ctx.check(acm_draw_points_rgb8(ctx.handle(), U.handle(), nullptr, r, g, b, img.ptr(), w, h));
    return img.download();
}
// util::compute_image_quality_metrics (image_quality.rs:254-324); `combined` (optional) receives the display image
inline ImageQualityMetrics compute_image_quality_metrics(const CameraModel& input_model, const CameraModel& output_model, const double* xyz_aos, size_t n,
                                                         uint32_t w, uint32_t h, const std::vector<uint8_t>* reference = nullptr,
                                                         std::vector<uint8_t>* combined = nullptr) {
    const Context& ctx = input_model.ctx();
    Points X(ctx, 3, xyz_aos, n);
    const size_t bytes = (size_t)w * h * 3;
    std::unique_ptr<DeviceImage> ref, comb;
    if (reference) ref.reset(new DeviceImage(ctx, bytes, reference->data()));
    if (combined) comb.reset(new DeviceImage(ctx, bytes));
    acm_camera ci = input_model.block(), co = output_model.block();
    acm_image_quality out{};
    ctx.check(acm_image_quality_metrics(ctx.handle(), &ci, &co, X.handle(), w, h, ref ? ref->ptr() : nullptr, comb ? comb->ptr() : nullptr, &out));
    if (combined) *combined = comb->download();
    return {out.psnr, out.ssim};
}

}  // namespace acm
