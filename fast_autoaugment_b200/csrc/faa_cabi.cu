// faa_cabi.cu - host side of the C ABI declared in include/faa_b200.h:
// policy compilation (level -> magnitude -> Pillow fixed-point / LUT / blend parameters),
// the MT19937 parity sampler, normalisation tables, device-table management and launches.
// There is NO CPU implementation of the pixel path in this library: every compute entry
// point fails with FAA_ERR_NO_DEVICE when no CUDA device is usable.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/faa_b200.h"
#include "faa_kernels.cuh"

using namespace faa;

static_assert(sizeof(faa_sample_t) == 16 && sizeof(Sample) == 16, "sample record is 16 bytes");
static_assert(sizeof(faa_box_t) == 8 && sizeof(Box) == 8, "box record is 8 bytes");
static_assert(sizeof(OpRec) == 32, "op record is 32 bytes");
static_assert(sizeof(faa_rng_t) == sizeof(RngCfg), "rng config layout");

// ------------------------------------------------------------------ errors --
static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const std::string& msg) { g_err = msg; return code; }
static int cuda_fail(cudaError_t e, const char* what) {
    return fail(FAA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(e__, #call); } while (0)

// --------------------------------------------------------------- op table --
struct OpInfo { const char* name; double low, high; int draw; };
// augment_list(for_autoaug=True): augmentations.py:156-182
static const OpInfo kOps[FAA_NUM_OPS] = {
    {"ShearX", -0.3, 0.3, FAA_DRAW_MIRROR},      {"ShearY", -0.3, 0.3, FAA_DRAW_MIRROR},
    {"TranslateX", -0.45, 0.45, FAA_DRAW_MIRROR}, {"TranslateY", -0.45, 0.45, FAA_DRAW_MIRROR},
    {"Rotate", -30, 30, FAA_DRAW_MIRROR},        {"AutoContrast", 0, 1, FAA_DRAW_NONE},
    {"Invert", 0, 1, FAA_DRAW_NONE},             {"Equalize", 0, 1, FAA_DRAW_NONE},
    {"Solarize", 0, 256, FAA_DRAW_NONE},         {"Posterize", 4, 8, FAA_DRAW_NONE},
    {"Contrast", 0.1, 1.9, FAA_DRAW_NONE},       {"Color", 0.1, 1.9, FAA_DRAW_NONE},
    {"Brightness", 0.1, 1.9, FAA_DRAW_NONE},     {"Sharpness", 0.1, 1.9, FAA_DRAW_NONE},
    {"Cutout", 0, 0.2, FAA_DRAW_BOX},            {"CutoutAbs", 0, 20, FAA_DRAW_BOX},
    {"Posterize2", 0, 4, FAA_DRAW_NONE},         {"TranslateXAbs", 0, 10, FAA_DRAW_MIRROR},
    {"TranslateYAbs", 0, 10, FAA_DRAW_MIRROR},
};

// ---------------------------------------------------------- compile helpers --
static inline int32_t fix16(double z) { return (int32_t)std::floor(z * 65536.0 + 0.5); }   // Pillow FIX()

// Python's round(x, 15): correctly rounded decimal round trip
static double py_round15(double x) {
    char buf[64];
    snprintf(buf, sizeof buf, "%.15f", x);
    return strtod(buf, nullptr);
}
// Python float %: result takes the sign of the divisor
static double py_fmod(double a, double b) {
    double r = std::fmod(a, b);
    if (r != 0.0 && ((r < 0.0) != (b < 0.0))) r += b;
    return r;
}
// ImagingScaleAffine axis table (Geometry.c): o = offset + scale*0.5, then o += scale per
// pixel, COORD(o) = o < 0 ? -1 : (int)o.  With unit scale the table is "i + shift", except
// that the repeatedly rounded accumulator may snap up to the next integer once (when
// offset+0.5 sits a few ulp below an integer): from index `brk` on the shift is shift+1.
// Returns false when the table is anything else.
static bool unit_scale_shift(int n, double offset, int32_t* shift, int32_t* brk) {
    double o = offset + 0.5;
    bool have = false; int32_t sh = 0, bk = INT32_MAX;
    std::vector<int32_t> tab(n);
    for (int i = 0; i < n; ++i) { tab[i] = (o < 0.0) ? INT32_MIN : (int32_t)o; o += 1.0; }
    for (int i = 0; i < n; ++i) {
        if (tab[i] == INT32_MIN) continue;
        int32_t d = tab[i] - i;
        if (!have) { sh = d; have = true; }
        else if (d == sh + 1 && bk == INT32_MAX) bk = i;
        else if (d != sh + (bk != INT32_MAX ? 1 : 0)) return false;
    }
    if (!have) { *shift = -2 * (int32_t)FAA_MAX_DIM; *brk = INT32_MAX; return true; }   // everything is fill
    for (int i = 0; i < n; ++i) {            // negative accumulator => Pillow skips the pixel
        if (tab[i] != INT32_MIN) continue;
        int32_t c = i + sh + (i >= bk ? 1 : 0);
        if (c >= 0 && c < n) return false;
    }
    *shift = sh; *brk = bk;
    return true;
}

struct Compiled { OpRec rec; int err; };   // err: 0 ok, FAA_ERR_UNKNOWN_OP, FAA_ERR_MAGNITUDE, FAA_ERR_UNSUPPORTED

static void set_affine(OpRec& r, const double m[6], int H, int W, int& err) {
    if (m[1] == 0.0 && m[3] == 0.0) {                     // Pillow: pure scale -> ImagingScaleAffine
        if (m[0] != 1.0 || m[4] != 1.0) { err = FAA_ERR_UNSUPPORTED; return; }
        int32_t dx, dy, bx, by;
        if (!unit_scale_shift(W, m[2], &dx, &bx) || !unit_scale_shift(H, m[5], &dy, &by)) { err = FAA_ERR_UNSUPPORTED; return; }
        if (dx == 0 && dy == 0 && bx == INT32_MAX && by == INT32_MAX) { r.kind = K_NONE; return; }
        r.kind = K_SHIFT; r.a[0] = dx; r.a[1] = dy; r.a[2] = bx; r.a[3] = by;
        return;
    }
    r.kind = K_AFFINE;                                    // Pillow affine_fixed
    r.a[0] = fix16(m[0]); r.a[1] = fix16(m[1]); r.a[2] = fix16(m[2] + m[0] * 0.5 + m[1] * 0.5);
    r.a[3] = fix16(m[3]); r.a[4] = fix16(m[4]); r.a[5] = fix16(m[5] + m[3] * 0.5 + m[4] * 0.5);
}

static void set_blend(OpRec& r, int kind, double v) {
    float a = (float)v;                                   // _blend passes a C float to ImagingBlend
    r.kind = kind;
    memcpy(&r.a[0], &a, 4);
    r.a[1] = !(a >= 0.0f && a <= 1.0f);
}

// apply_augment (augmentations.py:192-194) + the op's own parameter handling, at compile time
static Compiled compile_op(int op_id, double level, int sign, int H, int W) {
    Compiled c; memset(&c, 0, sizeof c);
    OpRec& r = c.rec; r.kind = K_NONE;
    if (op_id < 0 || op_id >= FAA_NUM_OPS) { c.err = FAA_ERR_UNKNOWN_OP; return c; }
    const OpInfo& info = kOps[op_id];
    r.draw = info.draw;
    double v = level * (info.high - info.low) + info.low;
    // the reference's per-op asserts (CutoutAbs' is commented out, augmentations.py:127)
    bool has_assert = !(op_id == FAA_AUTOCONTRAST || op_id == FAA_INVERT || op_id == FAA_EQUALIZE || op_id == FAA_CUTOUT_ABS);
    if (has_assert && !(info.low <= v && v <= info.high)) { c.err = FAA_ERR_MAGNITUDE; return c; }
    if (info.draw == FAA_DRAW_MIRROR && sign) v = -v;
    double m[6] = {1, 0, 0, 0, 1, 0};
    switch (op_id) {
    case FAA_SHEAR_X: m[1] = v; set_affine(r, m, H, W, c.err); break;                        // :17
    case FAA_SHEAR_Y: m[3] = v; set_affine(r, m, H, W, c.err); break;                        // :24
    case FAA_TRANSLATE_X: m[2] = v * (double)W; set_affine(r, m, H, W, c.err); break;        // :31-32
    case FAA_TRANSLATE_Y: m[5] = v * (double)H; set_affine(r, m, H, W, c.err); break;        // :39-40
    case FAA_TRANSLATE_X_ABS: m[2] = v; set_affine(r, m, H, W, c.err); break;                // :47
    case FAA_TRANSLATE_Y_ABS: m[5] = v; set_affine(r, m, H, W, c.err); break;                // :54
    case FAA_ROTATE: {                                                                        // :61 + PIL Image.rotate
        double angle = py_fmod(v, 360.0);
        if (angle == 0.0) break;                                                              // copy fast path
        if (angle == 180.0 || ((angle == 90.0 || angle == 270.0) && W == H)) { c.err = FAA_ERR_UNSUPPORTED; break; }
        double cx = W / 2.0, cy = H / 2.0;
        double t = -(angle * (M_PI / 180.0));                                                 // -math.radians(angle)
        m[0] = py_round15(std::cos(t)); m[1] = py_round15(std::sin(t)); m[2] = 0.0;
        m[3] = py_round15(-std::sin(t)); m[4] = py_round15(std::cos(t)); m[5] = 0.0;
        double t2 = m[0] * (-cx) + m[1] * (-cy) + m[2];
        double t5 = m[3] * (-cx) + m[4] * (-cy) + m[5];
        m[2] = t2 + cx; m[5] = t5 + cy;
        set_affine(r, m, H, W, c.err);
        break;
    }
    case FAA_AUTOCONTRAST: r.kind = K_AUTOCONTRAST; break;                                    // :65
    case FAA_EQUALIZE: r.kind = K_EQUALIZE; break;                                            // :73
    case FAA_INVERT: r.kind = K_LUT; r.a[0] = 0; r.a[1] = 0xFF; break;                        // :69
    case FAA_SOLARIZE: {                                                                      // :82  (i < v with float v)
        double th = std::ceil(v);
        r.kind = K_LUT; r.a[0] = (int32_t)(th < 0 ? 0 : th > 256 ? 256 : th); r.a[1] = 0xFF;
        break;
    }
    case FAA_POSTERIZE: case FAA_POSTERIZE2: {                                                // :87-88, :93-94
        int bits = (int)v;
        int mask = ~((1 << (8 - bits)) - 1) & 0xFF;
        r.kind = K_LUT; r.a[0] = 256; r.a[1] = mask;
        break;
    }
    case FAA_CONTRAST: set_blend(r, K_CONTRAST, v); break;                                    // :99
    case FAA_COLOR: set_blend(r, K_COLOR, v); break;                                          // :104
    case FAA_BRIGHTNESS: set_blend(r, K_BRIGHTNESS, v); break;                                // :109
    case FAA_SHARPNESS: set_blend(r, K_SHARPNESS, v); break;                                  // :114
    case FAA_CUTOUT: {                                                                        // :117-123
        if (v <= 0.0) { r.draw = FAA_DRAW_NONE; break; }                                      // returns before any draw
        double px = v * (double)W;
        r.kind = K_CUTOUT; memcpy(&r.a[0], &px, 8);
        break;
    }
    case FAA_CUTOUT_ABS: {                                                                    // :126-144
        if (v < 0.0) { r.draw = FAA_DRAW_NONE; break; }
        r.kind = K_CUTOUT; memcpy(&r.a[0], &v, 8);
        break;
    }
    }
    if (c.err) r.kind = K_NONE;
    return c;
}

// ------------------------------------------------------------------ policy --
struct DeviceTable { OpRec* d_ops = nullptr; };

struct faa_policy {
    int n_sub = 0, n_op = 0;
    std::vector<int32_t> op_ids;
    std::vector<double> probs, levels;
    std::mutex mu;
    std::map<std::pair<int, int>, std::vector<Compiled>> host_tables;   // (H,W) -> [n_sub][n_op][2]
    std::map<std::pair<int, int>, DeviceTable> dev_tables;
    double* d_probs = nullptr;
    float* d_norm = nullptr;            // [3][256]
    float norm_mean[3] = {-1e30f, 0, 0}, norm_std[3] = {0, 0, 0};
    float norm_host[768];
    bool fma_known[2] = {false, false}, fma_ok[2] = {false, false};   // [fp16, bf16]: does fmaf(u, scale, bias) round like the table?
    // scratch of faa_augment_host
    void* d_progs = nullptr; size_t d_progs_bytes = 0;
    void* d_order = nullptr;             // int32 [capacity of d_progs in images] (+ counters), two slots like d_progs
    // resolve-ahead: the decisions of the NEXT batch are resolved on a side stream while this batch's
    // pixels are computed; a call whose (rng, shapes, ...) key matches the speculation skips its resolve launch
    struct AheadKey { uint64_t seed, first_index; int32_t v[16]; };
    AheadKey ahead_key{}; bool ahead_valid = false; int ahead_slot = 0, cur_slot = 0;
    uint64_t last_first_index = 0; bool have_last = false; AheadKey last_key{};
    cudaStream_t ahead_stream = nullptr; cudaEvent_t ev_ahead = nullptr;
    void* d_scratch = nullptr; size_t d_scratch_bytes = 0;   // Sharpness->gather scratch images
    bool overlap_calls = false;          // faa_policy_set_overlap: consecutive calls on one stream may overlap (see augment_common)
    uint32_t done_target[2] = {0, 0};    // persistent chained steps: CTAs that have been launched on each program slot so far
    int sm_count = 0;
    bool has_sg = false;                 // some sub-policy has Sharpness followed by a geometric op
    void* d_in = nullptr; size_t d_in_bytes = 0;
    void* d_out = nullptr; size_t d_out_bytes = 0;
    void* h_in_stage = nullptr; size_t h_in_bytes = 0;
    void* h_out_stage = nullptr; size_t h_out_bytes = 0;
    cudaStream_t side[2] = {nullptr, nullptr};
    cudaStream_t light_stream = nullptr; cudaEvent_t ev_res = nullptr, ev_light = nullptr;
    cudaStream_t mid_stream = nullptr; cudaEvent_t ev_mid = nullptr;   // the mid kernel of a three-way split co-runs on its own stream
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    cudaEvent_t ev_host_done = nullptr; bool host_in_flight = false;   // faa_augment_host: last call's work (it owns d_in / stages)
    std::mutex call_mu;                  // launches of one policy are serialised (speculation state, slots, staging)
    const float* lighting_rgb = nullptr; int lighting_n = 0;       // Lighting offsets [n][3] (device) for the next launches, or null
    float* d_norm_img = nullptr; size_t d_norm_img_bytes = 0;      // per-image normalisation tables [n][3][256]
    int device = -1;                     // the device that owns every buffer / stream / event above (-1: none yet)
    int32_t ticket = 0;                  // chained steps: id of the last resolve launch
    int32_t ahead_ticket = 0;
    cudaStream_t chain_stream = nullptr; bool chain_live = false;   // the previous call was a chained step on this stream
    uintptr_t prev_out[2] = {0, 0}, prev_in[2] = {0, 0};            // byte ranges the previous chained step wrote / read
};

// All device state of a policy handle lives on ONE device: the one current at its first device call.
static int bind_device(faa_policy* p) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return fail(FAA_ERR_NO_DEVICE, "no current CUDA device"); }
    std::lock_guard<std::mutex> lk(p->mu);
    if (p->device < 0) p->device = dev;
    if (p->device != dev)
        return fail(FAA_ERR_VALUE, "policy handle is bound to device " + std::to_string(p->device) + " but the current device is " +
                    std::to_string(dev) + ": create one policy handle per device");
    return FAA_OK;
}

static const std::vector<Compiled>& host_table(faa_policy* p, int H, int W) {
    std::lock_guard<std::mutex> lk(p->mu);
    auto key = std::make_pair(H, W);
    auto it = p->host_tables.find(key);
    if (it != p->host_tables.end()) return it->second;
    std::vector<Compiled> t((size_t)p->n_sub * p->n_op * 2);
    for (int s = 0; s < p->n_sub; ++s)
        for (int j = 0; j < p->n_op; ++j)
            for (int sg = 0; sg < 2; ++sg) {
                size_t k = (size_t)s * p->n_op + j;
                t[k * 2 + sg] = compile_op(p->op_ids[k], p->levels[k], sg, H, W);
            }
    return p->host_tables.emplace(key, std::move(t)).first->second;
}

static int first_table_error(const std::vector<Compiled>& t, std::string& what) {
    for (size_t i = 0; i < t.size(); ++i)
        if (t[i].err) {
            what = "sub-policy " + std::to_string(i / 2) + " (flattened op index)";
            return t[i].err;
        }
    return 0;
}

extern "C" {

int faa_abi_version(void) { return FAA_ABI_VERSION; }
const char* faa_last_error(void) { return g_err.c_str(); }
uint64_t faa_launch_count(void) { return g_launches.load(); }

int faa_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int faa_op_id_from_name(const char* name) {
    if (!name) return -1;
    for (int i = 0; i < FAA_NUM_OPS; ++i) if (strcmp(name, kOps[i].name) == 0) return i;
    return -1;
}
const char* faa_op_name(int op_id) { return (op_id >= 0 && op_id < FAA_NUM_OPS) ? kOps[op_id].name : nullptr; }
int faa_op_range(int op_id, double* low, double* high) {
    if (op_id < 0 || op_id >= FAA_NUM_OPS) return fail(FAA_ERR_UNKNOWN_OP, "unknown op id");
    if (low) *low = kOps[op_id].low;
    if (high) *high = kOps[op_id].high;
    return FAA_OK;
}

int faa_policy_create(const int32_t* op_ids, const double* probs, const double* levels, int n_sub, int n_op,
                      faa_policy_t** out) {
    if (!op_ids || !probs || !levels || !out) return fail(FAA_ERR_VALUE, "null argument");
    if (n_sub <= 0 || n_sub > 65535) return fail(FAA_ERR_VALUE, "n_sub must be in [1, 65535]");
    if (n_op <= 0 || n_op > FAA_MAX_POLICY_OPS) return fail(FAA_ERR_VALUE, "n_op must be in [1, 8]");
    faa_policy* p = new faa_policy();
    p->n_sub = n_sub; p->n_op = n_op;
    size_t n = (size_t)n_sub * n_op;
    p->op_ids.assign(op_ids, op_ids + n);
    p->probs.assign(probs, probs + n);
    p->levels.assign(levels, levels + n);
    auto is_geo = [](int id) { return id == FAA_SHEAR_X || id == FAA_SHEAR_Y || id == FAA_TRANSLATE_X || id == FAA_TRANSLATE_Y ||
                                      id == FAA_ROTATE || id == FAA_TRANSLATE_X_ABS || id == FAA_TRANSLATE_Y_ABS; };
    for (int s = 0; s < n_sub && !p->has_sg; ++s)
        for (int j = 0; j + 1 < n_op; ++j)
            if (op_ids[(size_t)s * n_op + j] == FAA_SHARPNESS && is_geo(op_ids[(size_t)s * n_op + j + 1])) p->has_sg = true;
    *out = p;
    return FAA_OK;
}

int faa_policy_destroy(faa_policy_t* p) {
    if (!p) return FAA_OK;
    for (auto& kv : p->dev_tables) if (kv.second.d_ops) cudaFree(kv.second.d_ops);
    if (p->d_probs) cudaFree(p->d_probs);
    if (p->d_norm) cudaFree(p->d_norm);
    if (p->d_progs) cudaFree(p->d_progs);
    if (p->d_order) cudaFree(p->d_order);
    if (p->d_scratch) cudaFree(p->d_scratch);
    if (p->d_norm_img) cudaFree(p->d_norm_img);
    if (p->d_in) cudaFree(p->d_in);
    if (p->d_out) cudaFree(p->d_out);
    if (p->h_in_stage) cudaFreeHost(p->h_in_stage);
    if (p->h_out_stage) cudaFreeHost(p->h_out_stage);
    for (int i = 0; i < 2; ++i) {
        if (p->side[i]) cudaStreamDestroy(p->side[i]);
        if (p->ev_join[i]) cudaEventDestroy(p->ev_join[i]);
    }
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    if (p->ev_host_done) cudaEventDestroy(p->ev_host_done);
    if (p->light_stream) cudaStreamDestroy(p->light_stream);
    if (p->mid_stream) cudaStreamDestroy(p->mid_stream);
    if (p->ev_mid) cudaEventDestroy(p->ev_mid);
    if (p->ahead_stream) cudaStreamDestroy(p->ahead_stream);
    if (p->ev_ahead) cudaEventDestroy(p->ev_ahead);
    if (p->ev_res) cudaEventDestroy(p->ev_res);
    if (p->ev_light) cudaEventDestroy(p->ev_light);
    delete p;
    return FAA_OK;
}

int faa_policy_dims(const faa_policy_t* p, int* n_sub, int* n_op) {
    if (!p) return fail(FAA_ERR_VALUE, "null policy");
    if (n_sub) *n_sub = p->n_sub;
    if (n_op) *n_op = p->n_op;
    return FAA_OK;
}

static int check_shape(int h, int w) {
    if (h <= 0 || w <= 0 || h > FAA_MAX_DIM || w > FAA_MAX_DIM) return fail(FAA_ERR_VALUE, "image size out of range");
    return FAA_OK;
}

int faa_policy_compiled_op(faa_policy_t* p, int h, int w, int sub, int op, int sign, int32_t out8[8]) {
    if (!p || !out8) return fail(FAA_ERR_VALUE, "null argument");
    if (int e = check_shape(h, w)) return e;
    if (sub < 0 || sub >= p->n_sub || op < 0 || op >= p->n_op) return fail(FAA_ERR_VALUE, "index out of range");
    const Compiled& c = host_table(p, h, w)[((size_t)sub * p->n_op + op) * 2 + (sign ? 1 : 0)];
    memcpy(out8, &c.rec, 32);
    if (c.err) return fail(c.err, "op cannot be compiled (unknown op / magnitude out of range)");
    return FAA_OK;
}

int faa_policy_draw_kind(const faa_policy_t* p, int sub, int op) {
    if (!p || sub < 0 || sub >= p->n_sub || op < 0 || op >= p->n_op) return -1;
    int id = p->op_ids[(size_t)sub * p->n_op + op];
    if (id < 0 || id >= FAA_NUM_OPS) return -1;
    if (id == FAA_CUTOUT) {
        double v = p->levels[(size_t)sub * p->n_op + op] * (kOps[id].high - kOps[id].low) + kOps[id].low;
        if (v <= 0.0) return FAA_DRAW_NONE;
    }
    return kOps[id].draw;
}

int faa_cutout_box(const faa_policy_t* pc, int h, int w, int sub, int op, double ux, double uy, faa_box_t* out) {
    faa_policy* p = const_cast<faa_policy*>(pc);
    if (!p || !out) return fail(FAA_ERR_VALUE, "null argument");
    if (int e = check_shape(h, w)) return e;
    if (sub < 0 || sub >= p->n_sub || op < 0 || op >= p->n_op) return fail(FAA_ERR_VALUE, "index out of range");
    const Compiled& c = host_table(p, h, w)[((size_t)sub * p->n_op + op) * 2];
    if (c.err) return fail(c.err, "op cannot be compiled");
    if (c.rec.kind != K_CUTOUT) return fail(FAA_ERR_VALUE, "op draws no box");
    double v; memcpy(&v, &c.rec.a[0], 8);
    Box b = cutout_box(w, h, v, ux, uy);
    memcpy(out, &b, 8);
    return FAA_OK;
}

// ------------------------------------------------------------ MT19937 replay --
struct MT {
    uint32_t* s; uint32_t* pos;
    explicit MT(uint32_t st[625]) : s(st), pos(st + 624) {}
    void refill() {
        const uint32_t N = 624, M = 397, UP = 0x80000000u, LO = 0x7fffffffu, A = 0x9908b0dfu;
        uint32_t y; uint32_t kk;
        for (kk = 0; kk < N - M; ++kk) { y = (s[kk] & UP) | (s[kk + 1] & LO); s[kk] = s[kk + M] ^ (y >> 1) ^ ((y & 1u) ? A : 0u); }
        for (; kk < N - 1; ++kk) { y = (s[kk] & UP) | (s[kk + 1] & LO); s[kk] = s[kk + (M - N)] ^ (y >> 1) ^ ((y & 1u) ? A : 0u); }
        y = (s[N - 1] & UP) | (s[0] & LO); s[N - 1] = s[M - 1] ^ (y >> 1) ^ ((y & 1u) ? A : 0u);
        *pos = 0;
    }
    uint32_t u32() {
        if (*pos >= 624) refill();
        uint32_t y = s[(*pos)++];
        y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
        return y;
    }
    double real53() {   // CPython random.random() and numpy legacy random_sample(): same formula
        uint32_t a = u32() >> 5, b = u32() >> 6;
        return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0);
    }
    uint32_t below(uint32_t n) {   // CPython _randbelow_with_getrandbits
        int k = 32 - __builtin_clz(n);
        uint32_t r;
        do { r = u32() >> (32 - k); } while (r >= n);
        return r;
    }
};

int faa_sample_policy_mt(const faa_policy_t* pc, int batch, int h, int w, uint32_t py_state[625],
                         uint32_t np_state[625], faa_sample_t* out_samples, faa_box_t* out_boxes) {
    faa_policy* p = const_cast<faa_policy*>(pc);
    if (!p || !py_state || !np_state || !out_samples || !out_boxes) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0) return fail(FAA_ERR_VALUE, "negative batch");
    if (int e = check_shape(h, w)) return e;
    if (py_state[624] > 624 || np_state[624] > 624) return fail(FAA_ERR_VALUE, "bad MT19937 position");
    const std::vector<Compiled>& tab = host_table(p, h, w);
    MT py(py_state), np(np_state);
    for (int i = 0; i < batch; ++i) {
        faa_sample_t s; memset(&s, 0, sizeof s);
        uint32_t sub = py.below((uint32_t)p->n_sub);                          // random.choice, data.py:259
        s.sub = (uint16_t)sub;
        for (int j = 0; j < p->n_op; ++j) {
            faa_box_t& bx = out_boxes[(size_t)i * p->n_op + j];
            bx.x0 = bx.y0 = 0; bx.x1 = bx.y1 = -1;
            size_t k = (size_t)sub * p->n_op + j;
            if (p->probs[k] < 0.0) continue;                                   // padding slot of a ragged sub-policy: no draw
            if (py.real53() > p->probs[k]) continue;                           // data.py:261
            const Compiled& c0 = tab[k * 2];
            if (c0.err) return fail(c0.err, std::string("applied op is invalid: ") +
                                    (c0.err == FAA_ERR_UNKNOWN_OP ? "unknown op" : "magnitude out of range / unsupported"));
            s.gate |= (uint8_t)(1u << j);
            if (c0.rec.draw == FAA_DRAW_MIRROR) {
                if (py.real53() > 0.5) s.sign |= (uint8_t)(1u << j);           // augmentations.py:15 ...
            } else if (c0.rec.draw == FAA_DRAW_BOX) {
                double ux = np.real53(), uy = np.real53();                     // augmentations.py:131-132
                double v; memcpy(&v, &c0.rec.a[0], 8);
                Box b = cutout_box(w, h, v, ux, uy);
                memcpy(&bx, &b, 8);
            }
        }
        out_samples[i] = s;
    }
    return FAA_OK;
}

// ------------------------------------------------------------ device tables --
static int ensure_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(FAA_ERR_NO_DEVICE, "no CUDA device available: fast_autoaugment_b200 has no CPU fallback");
    }
    return FAA_OK;
}

static int device_table(faa_policy* p, int H, int W, bool need_valid, const OpRec** d_ops) {
    const std::vector<Compiled>& t = host_table(p, H, W);
    if (need_valid) {
        std::string what;
        if (int e = first_table_error(t, what))
            return fail(e, "policy contains an op that cannot run (" + what + "): unknown op or magnitude out of range");
    }
    std::lock_guard<std::mutex> lk(p->mu);
    auto key = std::make_pair(H, W);
    auto it = p->dev_tables.find(key);
    if (it == p->dev_tables.end()) {
        std::vector<OpRec> flat(t.size());
        for (size_t i = 0; i < t.size(); ++i) flat[i] = t[i].rec;
        DeviceTable d;
        CK(cudaMalloc(&d.d_ops, flat.size() * sizeof(OpRec)));
        CK(cudaMemcpy(d.d_ops, flat.data(), flat.size() * sizeof(OpRec), cudaMemcpyHostToDevice));
        it = p->dev_tables.emplace(key, d).first;
    }
    if (!p->d_probs) {
        CK(cudaMalloc(&p->d_probs, p->probs.size() * sizeof(double)));
        CK(cudaMemcpy(p->d_probs, p->probs.data(), p->probs.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    *d_ops = it->second.d_ops;
    return FAA_OK;
}

// ToTensor + Normalize exactly as torch computes them in fp32 (data.py:42-43):
// x = u8 / 255 ; (x - mean) / std.  Also decides whether one fused multiply-add reproduces
// the rounded result for every byte value in the requested output dtype.
static uint16_t bits16(int dtype, float v) {
    if (dtype == FAA_F16) { __half h = __float2half_rn(v); return __half_as_ushort(h); }
    __nv_bfloat16 b = __float2bfloat16_rn(v); return __bfloat16_as_ushort(b);
}

static int normalisation(faa_policy* p, const faa_tail_t* tail, AugParams& P, bool& use_tab, cudaStream_t stream) {
    bool same = true;
    for (int c = 0; c < 3; ++c) same = same && p->norm_mean[c] == tail->mean[c] && p->norm_std[c] == tail->std[c];
    if (!p->d_norm) { CK(cudaMalloc(&p->d_norm, 768 * sizeof(float))); same = false; }
    if (!same) {
        for (int c = 0; c < 3; ++c) {
            if (!(tail->std[c] != 0.0f)) return fail(FAA_ERR_VALUE, "std must be non-zero");
            for (int u = 0; u < 256; ++u) {
                volatile float x = (float)u / 255.0f;
                volatile float y = x - tail->mean[c];
                volatile float z = y / tail->std[c];
                p->norm_host[c * 256 + u] = z;
            }
            p->norm_mean[c] = tail->mean[c]; p->norm_std[c] = tail->std[c];
        }
        CK(cudaMemcpyAsync(p->d_norm, p->norm_host, 768 * sizeof(float), cudaMemcpyHostToDevice, stream));
    }
    P.norm_tab = p->d_norm;
    if (!same) p->fma_known[0] = p->fma_known[1] = false;
    const bool half_out = tail->out_dtype == FAA_F16 || tail->out_dtype == FAA_BF16;
    const int slot = tail->out_dtype == FAA_BF16 ? 1 : 0;
    bool fma_ok = half_out;
    for (int c = 0; c < 3; ++c) {
        double sc = 1.0 / (255.0 * (double)tail->std[c]);
        double bi = -(double)tail->mean[c] / (double)tail->std[c];
        P.scale[c] = (float)sc; P.bias[c] = (float)bi;
    }
    if (half_out && p->fma_known[slot]) {
        fma_ok = p->fma_ok[slot];                           // (768 conversions per call are a visible part of a small step)
    } else if (half_out) {
        for (int c = 0; c < 3 && fma_ok; ++c)
            for (int u = 0; u < 256 && fma_ok; ++u) {
                float f = fmaf((float)u, P.scale[c], P.bias[c]);
                if (bits16(tail->out_dtype, f) != bits16(tail->out_dtype, p->norm_host[c * 256 + u])) fma_ok = false;
            }
        p->fma_known[slot] = true; p->fma_ok[slot] = fma_ok;
    }
    use_tab = !fma_ok;
    return FAA_OK;
}

static int out_elem_size(int dtype) { return dtype == FAA_F32 ? 4 : dtype == FAA_U8_HWC ? 1 : 2; }

// RandomCrop offsets travel as int8 (faa_sample_t): ranges that do not fit are refused, never silently changed
static int check_crop(int h, int w, const faa_tail_t* tail, int crop_pad) {
    const int span_y = h + 2 * crop_pad - tail->out_h, span_x = w + 2 * crop_pad - tail->out_w;
    if (span_y < 0 || span_x < 0)
        return fail(FAA_ERR_VALUE, "Required crop size is larger than the (padded) input image size");   // torchvision's message
    if (crop_pad > 127 || span_y - crop_pad > 127 || span_x - crop_pad > 127)
        return fail(FAA_ERR_UNSUPPORTED, "RandomCrop offsets beyond +-127 pixels are not supported (int8 records): crop on the host side");
    return FAA_OK;
}

static int check_tail(const faa_tail_t* tail) {
    if (!tail) return fail(FAA_ERR_VALUE, "null tail");
    if (tail->out_h <= 0 || tail->out_w <= 0 || tail->out_h > FAA_MAX_DIM || tail->out_w > FAA_MAX_DIM)
        return fail(FAA_ERR_VALUE, "output size out of range");
    if (tail->out_dtype < 0 || tail->out_dtype > FAA_U8_HWC) return fail(FAA_ERR_VALUE, "bad out_dtype");
    return FAA_OK;
}

int faa_sample_philox(faa_policy_t* p, int batch, int h, int w, const faa_tail_t* tail, const faa_rng_t* rng,
                      faa_sample_t* d_samples, faa_box_t* d_boxes, void* stream) {
    if (!p || !rng || !d_samples || !d_boxes) return fail(FAA_ERR_VALUE, "null argument");
    if (int e = check_shape(h, w)) return e;
    if (int e = check_tail(tail)) return e;
    if (int e = check_crop(h, w, tail, rng->crop_pad > 0 ? rng->crop_pad : 0)) return e;
    if (int e = ensure_device()) return e;
    if (int e = bind_device(p)) return e;
    const OpRec* d_ops = nullptr;
    if (int e = device_table(p, h, w, true, &d_ops)) return e;
    ResolveParams R; memset(&R, 0, sizeof R);
    R.ops = d_ops; R.probs = p->d_probs; memcpy(&R.rng, rng, sizeof(RngCfg));
    R.samples_out = reinterpret_cast<Sample*>(d_samples); R.boxes_out = reinterpret_cast<Box*>(d_boxes);
    R.first = 0; R.n = batch; R.H = h; R.W = w; R.out_h = tail->out_h; R.out_w = tail->out_w;
    R.n_sub = p->n_sub; R.n_op = p->n_op; R.op_base = 0; R.apply_tail = 1;
    CK(launch_resolve(R, (cudaStream_t)stream));
    if (batch > 0) g_launches++;
    return FAA_OK;
}

static int augment_common(faa_policy_t* p, const uint8_t* d_in_all, int n_all, int first, void* d_out, int batch,
                          int h, int w, const faa_tail_t* tail, const faa_sample_t* d_samples,
                          const faa_box_t* d_boxes, const faa_rng_t* rng, int op_base, const int32_t* d_partner,
                          float lam, float oml, int apply_tail, bool allow_ahead, void* stream_v, int in_mod = 0) {
    if (!p || (!d_in_all && batch > 0) || (!d_out && batch > 0)) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0 || first < 0 || first + batch > n_all) return fail(FAA_ERR_VALUE, "bad batch range");
    if (batch > 65535) return fail(FAA_ERR_UNSUPPORTED, "at most 65535 images per call (one grid row per image): split the batch");
    if (int e = check_shape(h, w)) return e;
    if (int e = check_tail(tail)) return e;
    if (!d_samples && !rng) return fail(FAA_ERR_VALUE, "need either resolved samples or an rng config");
    if (rng && !d_samples && apply_tail) { if (int e = check_crop(h, w, tail, rng->crop_pad > 0 ? rng->crop_pad : 0)) return e; }
    if (op_base < 0 || op_base >= p->n_op) return fail(FAA_ERR_VALUE, "op_base out of range");
    if (tail->out_dtype == FAA_U8_HWC && d_partner) return fail(FAA_ERR_UNSUPPORTED, "mixup needs a float output");
    if (int e = ensure_device()) return e;
    if (batch == 0) return FAA_OK;
    if (int e = bind_device(p)) return e;
    cudaStream_t stream = (cudaStream_t)stream_v;
    const OpRec* d_ops = nullptr;
    // resolved samples can only reference ops the host sampler validated; Philox can pick anything
    if (int e = device_table(p, h, w, d_samples == nullptr, &d_ops)) return e;
    {   // per-image program buffer (grown, never shrunk; stream-ordered reuse)
        std::lock_guard<std::mutex> lk(p->mu);
        size_t need = (size_t)n_all * sizeof(Prog);
        if (p->d_progs_bytes < need) {
            if (p->d_progs) {
                CK(cudaStreamSynchronize(stream));
                if (p->ahead_stream) CK(cudaStreamSynchronize(p->ahead_stream));
                CK(cudaFree(p->d_progs)); CK(cudaFree(p->d_order));
                p->d_progs = p->d_order = nullptr; p->d_progs_bytes = 0;
            }
            need = need < 65536 ? 65536 : need * 2;
            CK(cudaMalloc(&p->d_progs, 2 * need));                                                // two slots (resolve-ahead)
            CK(cudaMalloc(&p->d_order, 2 * (4 * (need / sizeof(Prog)) * sizeof(int32_t) + 32)));  // order + 2 counters per launch + ready words, x2
            CK(cudaMemset(p->d_order, 0, 2 * (4 * (need / sizeof(Prog)) * sizeof(int32_t) + 32)));
            p->d_progs_bytes = need;
            p->ahead_valid = false;
            p->done_target[0] = p->done_target[1] = 0;      // (the completion counters live in d_order and start at zero)
        }
    }
    // geometry of the pixel launch (needed by the resolve step: allow_mat)
    AugParams P; memset(&P, 0, sizeof P);
    P.in = d_in_all; P.out = d_out;
    P.partner = d_partner;
    P.B = batch; P.H = h; P.W = w; P.out_h = tail->out_h; P.out_w = tail->out_w; P.first = first; P.in_mod = in_mod;
    P.use_zero_box = (tail->use_zero_box && apply_tail) ? 1 : 0;
    P.lam = lam; P.one_minus_lam = oml;
    P.bands = pick_bands(h, w, tail->out_h, tail->out_w);
    static const bool lpt_off = [] { const char* e = getenv("FAA_LPT"); return e && e[0] == '0'; }();
    // TMA band staging needs 16-byte aligned image bases and a band that fits shared memory
    // (crop_pad only sizes the staged band; rows outside it are read from global memory)
    P.crop_pad = tail->crop_pad > 0 ? tail->crop_pad : 0;
    if (rng && rng->crop_pad > P.crop_pad) P.crop_pad = rng->crop_pad;
    if (P.crop_pad > h) P.crop_pad = h;
    P.band_cap = (int32_t)band_capacity(P.bands, h, w, tail->out_h, P.crop_pad);
    const size_t img_bytes = (size_t)h * w * 3;
    const int nsrc = d_partner ? 2 : 1;
    static const bool stage_off = [] { const char* e = getenv("FAA_STAGE"); return e && e[0] == '0'; }();
    static const bool mat_off = [] { const char* e = getenv("FAA_MAT"); return e && e[0] == '0'; }();
    static const bool pdl_off = [] { const char* e = getenv("FAA_PDL"); return e && e[0] == '0'; }();
    P.stage = (!stage_off && img_bytes % 16 == 0 && ((uintptr_t)d_in_all % 16) == 0 &&
               (size_t)P.band_cap * nsrc <= 150 * 1024) ? 1 : 0;
    if (!P.stage) P.band_cap = 0;
    {   // per-kernel band geometry and fastdiv reciprocals (host side: no divisions in the kernels)
        fill_geom(P.geo[0], P.bands, h, w, tail->out_h, P.crop_pad, P.stage != 0);
        int lb = P.bands;
        if (P.bands == 8) {
            // the light kernel needs no cluster, so any band count works: take the one in 5..8 whose
            // quads-per-CTA fills whole 256-thread iterations best (224x224: 7 bands = exactly 7 iterations)
            const int qpr = (tail->out_w + 3) / 4;
            double best = -1.0;
            for (int b = 8; b >= 5; --b) {
                const int rows = (tail->out_h + b - 1) / b;
                const int quads = rows * qpr, iters = (quads + 255) / 256;
                const double eff = (double)quads / (iters * 256.0) * ((double)tail->out_h / (rows * b));
                if (eff > best + 0.02) { best = eff; lb = b; }
            }
        }
        static const int light_bands = [] { const char* e = getenv("FAA_LIGHT_BANDS"); return e ? atoi(e) : 0; }();
        if (light_bands >= 1 && light_bands <= 8 && light_bands <= h && light_bands <= tail->out_h) lb = light_bands;
        fill_geom(P.geo[1], lb, h, w, tail->out_h, P.crop_pad, P.stage != 0 && (size_t)band_capacity(lb, h, w, tail->out_h, P.crop_pad) <= 100 * 1024);
        auto rcp = [](uint32_t d) { return d <= 1 ? 0u : (uint32_t)((0x100000000ull + d - 1) / d); };
        P.rcp_out_qpr = rcp((uint32_t)(tail->out_w + 3) / 4); P.rcp_w = rcp((uint32_t)w); P.rcp_wq = rcp((uint32_t)w / 4);
        P.rcp_opr = (w & 7) ? 0u : rcp((uint32_t)w / 8);
        static const bool oct_off = [] { const char* e = getenv("FAA_OCTETS"); return e && e[0] == '0'; }();
        P.octets = (!oct_off && (w & 7) == 0 && tail->out_w == w && tail->out_h == h &&
                    ((uintptr_t)d_out % 16) == 0 && P.stage) ? 1 : 0;          // (uint8 HWC included: 24-byte octets, 8-byte aligned)
    }
    // materialisation chunk: as many rows as fit ~16 KB, at least 3 (single-source launches only)
    {
        // big enough to keep a whole band (+ halo, + crop slack) resident when that is <= 24 KB, else ~16 KB chunks
        const int pitch = w * 3;
        const int band_rows = (h + P.bands - 1) / P.bands + 2 + 2 * P.crop_pad;
        int rows = (band_rows * pitch <= 24576) ? band_rows : 16384 / pitch;
        if (rows > h + 2) rows = h + 2;
        P.mat_cap = (!mat_off && !d_partner && rows >= 3) ? ((rows * pitch + 32 + 15) & ~15) : 0;   // + 2 guard bands
    }
    P.pdl = pdl_off ? 0 : 1;
    // launch 1: decisions -> programs (the whole pool when partners may be anywhere in it)
    ResolveParams R; memset(&R, 0, sizeof R);
    R.ops = d_ops; R.probs = p->d_probs;
    R.samples = reinterpret_cast<const Sample*>(d_samples); R.boxes = reinterpret_cast<const Box*>(d_boxes);
    if (rng) memcpy(&R.rng, rng, sizeof(RngCfg));
    R.first = d_partner ? 0 : first; R.n = d_partner ? n_all : batch;
    R.H = h; R.W = w; R.out_h = tail->out_h; R.out_w = tail->out_w;
    R.n_sub = p->n_sub; R.n_op = p->n_op; R.op_base = op_base; R.apply_tail = apply_tail;
    R.allow = P.mat_cap > 0 ? 1 : 0;
    static const bool split_off = [] { const char* e = getenv("FAA_SPLIT"); return e && e[0] == '0'; }();
    static const bool ahead_off = [] { const char* e = getenv("FAA_AHEAD"); return e && e[0] == '0'; }();
    const bool use_order = !(d_partner || lpt_off);
    // (small launches are launch-latency bound: one pixel kernel is faster there)
    size_t split_min = (size_t)4 << 20;                   // pixels per launch from which two pixel kernels pay off
    if (const char* e = getenv("FAA_SPLIT_MIN")) split_min = (size_t)strtoull(e, nullptr, 10);   // tests: force either path
    // (uint8 HWC output - the Mixup exchange format - splits when the lean octet paths can write it)
    const bool use_split = use_order && !split_off && (tail->out_dtype != FAA_U8_HWC || (P.octets && P.crop_pad == 0 && apply_tail)) &&
                           (size_t)batch * h * w >= split_min;
    R.split = use_split ? 1 : 0;
    // Chained steps (default; FAA_CHAIN=0 selects the event schedule): resolve(N+1), [cluster(N),] mid(N), light(N) all on the
    // caller's stream with programmatic dependent launches, no events and no side streams.  Consecutive steps
    // overlap (the next step's CTAs fill the slots the previous step's tail frees); the only true dependency -
    // programs written by the resolve kernel - is a ticket word the pixel kernels poll.  FAA_CHAIN=0: the
    // two-stream schedule with events (light kernel on the caller's stream, cluster kernel on a priority stream).
    int chain_mode = 1;                                   // measured (profiles/r02_schedules.txt): 62.4 us chained vs 65.6 us with events
    if (const char* e = getenv("FAA_CHAIN")) chain_mode = atoi(e);
    // (launches too small to split are chained as well: resolve(N+1), cluster(N) - their step is bound by kernel latencies,
    //  which only overlap across steps on one stream; uint8 output stays on the event schedule)
    static const bool chain_small_off = [] { const char* e = getenv("FAA_CHAIN_SMALL"); return e && e[0] == '0'; }();
    const bool chain_small = !use_split && !chain_small_off && use_order && tail->out_dtype != FAA_U8_HWC;
    const bool use_chain = chain_mode != 0 && (use_split || chain_small) && allow_ahead && rng && !d_samples && !d_partner &&
                           !(getenv("FAA_AHEAD") && getenv("FAA_AHEAD")[0] == '0');
    // Three-way split: statistics-LUT and Sharpness programs run in the lean mid kernel.
    // Needs the geometry its paths assume: float planes of the image's own size, no crop, W % 4 == 0, staged bands.
    static const bool mid_off = [] { const char* e = getenv("FAA_MID"); return e && e[0] == '0'; }();
    const bool use_mid = use_split && !mid_off && P.stage && (w & 3) == 0 && tail->out_w == w && tail->out_h == h &&
                         P.crop_pad == 0 && ((uintptr_t)d_out % 16) == 0;
    if (use_mid) R.split = 2;
    if (use_split && P.octets && P.crop_pad == 0) R.allow |= 4;     // the lean gather paths exist in this launch
    // program / schedule buffers come in two slots; a slot = progs[cap] + order[cap] + counters[2 cap] + ready[cap]
    const size_t cap_imgs = p->d_progs_bytes / sizeof(Prog);
    auto bind_slot = [&](int slot, ResolveParams& r, AugParams* a) {
        Prog* progs = reinterpret_cast<Prog*>((uint8_t*)p->d_progs + (size_t)slot * p->d_progs_bytes);
        int32_t* order = reinterpret_cast<int32_t*>(p->d_order) + (size_t)slot * (4 * cap_imgs + 8);
        // the segment counters of a split launch live behind the order array, indexed by `first` so that
        // concurrent chunk launches do not share them (same for the ready word)
        int32_t* counter = order + cap_imgs + 2 * (size_t)first;
        int32_t* ready = order + 3 * cap_imgs + first;
        r.progs = progs; r.order = use_order ? order : nullptr; r.n_heavy = use_split ? counter : nullptr;
        r.ready = use_chain ? ready : nullptr;
        if (a) {
            a->progs = progs; a->order = use_order ? order : nullptr; a->n_heavy = use_split ? counter : nullptr;
            a->ready = use_chain ? ready : nullptr;
        }
    };
    // scratch images: Sharpness -> gather programs of the cluster kernel, every Sharpness-first two-op program of the mid kernel
    // Persistent mid / light kernels (chained schedule only; FAA_PERSIST=0 keeps one CTA row per image): rows loop over
    // their entries, all CTAs of a kernel are resident at once, so it releases its dependents immediately and consecutive
    // kernels - and steps - overlap for their whole length.  What the early release no longer orders is ordered explicitly:
    // program slots by completion counters the next resolve kernel of the slot waits for, scratch images by a copy per slot.
    static const bool persist_off = [] { const char* e = getenv("FAA_PERSIST"); return e && e[0] == '0'; }();
    const bool persist = use_chain && !persist_off;
    // The copy of slot 1 starts at a fixed half of the allocation, not behind this call's n_all images: the resolve kernel of
    // a slot only waits for that slot's previous readers, so after a batch-size change a slot's scratch must not move onto
    // the images the other slot's step - two steps back, possibly still running - reads.
    size_t scratch_half = 0;
    if ((p->has_sg || use_mid) && !d_partner && (w & 3) == 0) {
        const size_t scratch_slot_bytes = ((size_t)n_all * img_bytes + 255) & ~(size_t)255;
        const size_t need = scratch_slot_bytes * (persist ? 2 : 1);
        if (p->d_scratch_bytes < need) {
            if (p->d_scratch) { CK(cudaStreamSynchronize(stream)); CK(cudaFree(p->d_scratch)); p->d_scratch = nullptr; p->d_scratch_bytes = 0; }
            CK(cudaMalloc(&p->d_scratch, need));
            p->d_scratch_bytes = need;
        }
        P.scratch = (uint8_t*)p->d_scratch;
        scratch_half = (p->d_scratch_bytes / 2) & ~(size_t)255;      // >= scratch_slot_bytes whenever persist
        R.allow |= 2;
    }
    // With the lean gathers (allow bit 2) and a scratch image (bit 1) every program of a three-way split is light or mid
    // (faa_core.cuh prog_is_light / prog_is_mid cover all class combinations; tests/test_gpu_fastpaths.py runs every ordered
    // op pair through this schedule): the cluster kernel has nothing to do and is not launched.  FAA_HEAVY=1 launches it anyway.
    static const bool heavy_always = [] { const char* e = getenv("FAA_HEAVY"); return e && e[0] == '1'; }();
    const bool no_heavy = use_mid && (R.allow & 6) == 6 && P.mat_cap > 0 && !heavy_always;
    bool use_tab = false;
    if (tail->out_dtype != FAA_U8_HWC) { if (int e = normalisation(p, tail, P, use_tab, stream)) return e; }
    else { for (int c = 0; c < 3; ++c) { P.scale[c] = 1.0f; P.bias[c] = 0.0f; } }      // lean paths: the byte value itself
    if (p->lighting_rgb && tail->out_dtype != FAA_U8_HWC && apply_tail) {
        // Lighting (augmentations.py:197-215): one normalisation table per image, built on the stream in torch's fp32 order
        if (d_partner) return fail(FAA_ERR_UNSUPPORTED, "Lighting together with fused Mixup is not supported");
        if (p->lighting_n != n_all) return fail(FAA_ERR_VALUE, "faa_policy_set_lighting was given a different number of images");
        const size_t need = (size_t)n_all * 768 * sizeof(float);
        if (p->d_norm_img_bytes < need) {
            if (p->d_norm_img) { CK(cudaStreamSynchronize(stream)); CK(cudaFree(p->d_norm_img)); p->d_norm_img = nullptr; p->d_norm_img_bytes = 0; }
            CK(cudaMalloc(&p->d_norm_img, need));
            p->d_norm_img_bytes = need;
        }
        CK(launch_lighting_tables(p->lighting_rgb, p->d_norm_img, n_all, tail->mean, tail->std, stream));
        g_launches++;
        P.norm_tab = p->d_norm_img; P.norm_stride = 768;
        use_tab = true;
    }
    // fused Mixup mixes the fp32 normalised values before the output rounding: the fma shortcut is only proven to round
    // like the exact value for a DIRECT fp16 / bf16 store, so two-source launches always take the exact table
    if (d_partner) use_tab = true;
    // Self-resolving launch (FAA_SELF=0 turns it off): a launch of tiny images is bound by kernel latencies and by the
    // host's launch rate, not by bytes.  Thread 0 of every CTA draws its image's decisions and builds the program itself
    // (same Philox counters, same build_prog): ONE kernel per step, no program array, no ticket - consecutive steps have
    // no dependency left and overlap through programmatic dependent launch.
    static const bool self_off = [] { const char* e = getenv("FAA_SELF"); return e && e[0] == '0'; }();
    if (!use_split && !self_off && rng && !d_samples && !d_partner && (size_t)h * w <= 4096) {     // (tiny images: see below)
        const uintptr_t in0 = (uintptr_t)d_in_all + (in_mod ? 0 : (size_t)first * img_bytes),
                        in1 = in0 + (size_t)(in_mod ? in_mod : batch) * img_bytes;
        const uintptr_t out0 = (uintptr_t)d_out, out1 = out0 + (size_t)batch * tail->out_h * tail->out_w * 3 * out_elem_size(tail->out_dtype);
        auto overlap = [](uintptr_t a0, uintptr_t a1, const uintptr_t b[2]) { return a0 < b[1] && b[0] < a1; };
        const bool overlap_ok = p->overlap_calls && p->chain_live && p->chain_stream == stream && !overlap(in0, in1, p->prev_out) &&
                                !overlap(out0, out1, p->prev_out) && !overlap(out0, out1, p->prev_in) && !P.norm_stride;
        AugParams Ps = P;
        Ps.progs = nullptr; Ps.order = nullptr; Ps.n_heavy = nullptr; Ps.ready = nullptr; Ps.done = nullptr; Ps.grid_y = 0;
        Ps.self_resolve = 1;
        Ps.sr_ops = d_ops; Ps.sr_probs = p->d_probs; memcpy(&Ps.sr_rng, rng, sizeof(RngCfg));
        Ps.sr_n_sub = p->n_sub; Ps.sr_n_op = p->n_op; Ps.sr_op_base = op_base; Ps.sr_apply_tail = apply_tail; Ps.sr_allow = R.allow;
        // chain = 1: no griddepcontrol.wait (nothing of the previous kernel is consumed), dependents released once the CTA has
        // its program; a step that touches the previous step's buffers is launched as a plain stream-ordered kernel instead
        Ps.chain = overlap_ok ? 1 : 0; Ps.pdl = 0;
        // Only for tiny images (CIFAR): there the one-block resolve kernel is as long as the pixel kernel; for larger images
        // every band CTA would repeat ~10 us of serial work (measured: 224x224 b2048 uint8 launches 0.90 -> 0.97 ms).
        // Sharpness -> gather programs are evaluated lazily instead of through the scratch image - the last thing consecutive
        // steps shared - and every CTA releases the next step at once (chain = 3).
        Ps.sr_allow &= ~2; Ps.scratch = nullptr;
        if (overlap_ok) Ps.chain = 3;
        CK(launch_augment(Ps, tail->out_dtype, use_tab, 0, stream));
        g_launches++;
        p->ahead_valid = false;
        p->chain_live = true; p->chain_stream = stream;
        p->prev_in[0] = in0; p->prev_in[1] = in1; p->prev_out[0] = out0; p->prev_out[1] = out1;
        return FAA_OK;
    }
    // resolve-ahead: did the previous call already resolve exactly this batch on the side stream?
    const bool spec_ok = allow_ahead && !ahead_off && rng && !d_samples && !d_partner;
    faa_policy::AheadKey key; memset(&key, 0, sizeof key);
    if (spec_ok) {
        key.seed = rng->seed; key.first_index = rng->first_index;
        const int32_t v[16] = {batch, n_all, first, h, w, tail->out_h, tail->out_w, op_base, apply_tail, R.allow, R.split,
                               rng->crop_pad, rng->hflip, rng->zero_box_len, (use_order ? 1 : 0) | (in_mod << 1), (use_chain ? 1 : 0) | (P.norm_stride ? 2 : 0)};
        memcpy(key.v, v, sizeof v);
    }
    auto set_mid_geometry = [&](AugParams& a) {
        int mb = P.bands;                                   // halve the band count while a band (+ halo) stays <= 80 KB (2 CTAs / SM)
        while (mb > 1 && band_capacity(mb / 2, h, w, tail->out_h, 0) <= 80 * 1024) mb /= 2;
        static const int mid_bands = [] { const char* e = getenv("FAA_MID_BANDS"); return e ? atoi(e) : 0; }();
        if (mid_bands >= 1 && mid_bands <= 8 && (mid_bands & (mid_bands - 1)) == 0 && mid_bands <= h) mb = mid_bands;
        a.bands = mb;
        fill_geom(a.geo[0], mb, h, w, tail->out_h, 0, true);
        a.band_cap = a.geo[0].band_cap; a.mat_cap = 0;
    };
    const bool hit = spec_ok && p->ahead_valid && memcmp(&key, &p->ahead_key, sizeof key) == 0;
    int slot = p->cur_slot;
    if (use_chain) {
        // ---- chained schedule -------------------------------------------------------------------------
        // A step may only overlap the previous one if it neither reads what that step wrote nor writes what it
        // read or wrote (and follows it on the same stream); otherwise its first kernel is a plain dependent launch.
        const uintptr_t in0 = (uintptr_t)d_in_all + (in_mod ? 0 : (size_t)first * img_bytes),
                        in1 = in0 + (size_t)(in_mod ? in_mod : batch) * img_bytes;
        const uintptr_t out0 = (uintptr_t)d_out, out1 = out0 + (size_t)batch * tail->out_h * tail->out_w * 3 * out_elem_size(tail->out_dtype);
        auto overlap = [](uintptr_t a0, uintptr_t a1, const uintptr_t b[2]) { return a0 < b[1] && b[0] < a1; };
        // ... and only if the caller has promised that this call's inputs were complete before the previous call was issued
        // (faa_policy_set_overlap / faa_augment_many): a kernel launched with programmatic serialization that does not execute
        // griddepcontrol.wait has no visibility guarantee for what the kernel right in front of it wrote, and that kernel
        // may be the producer of this batch (a gather, a copy).  Within a call every kernel only consumes what its own
        // call's first - stream-ordered - kernel already waited for.
        bool overlap_ok = p->overlap_calls && p->chain_live && p->chain_stream == stream && !overlap(in0, in1, p->prev_out) &&
                          !overlap(out0, out1, p->prev_out) && !overlap(out0, out1, p->prev_in);
        AugParams Pc = P;
        Pc.chain = persist ? 2 : 1; Pc.pdl = 0;
        // completion counter of a slot: the first spare word behind its order / counters / ready arrays
        auto done_word = [&](int s) { return reinterpret_cast<uint32_t*>(reinterpret_cast<int32_t*>(p->d_order) + (size_t)s * (4 * cap_imgs + 8) + 4 * cap_imgs); };
        auto wait_for_slot = [&](int s, ResolveParams& r) {
            r.wait_done = persist ? done_word(s) : nullptr; r.wait_target = p->done_target[s];
        };
        if (hit) {
            slot = p->ahead_slot;
            Pc.ticket = p->ahead_ticket;
            bind_slot(slot, R, &Pc);
        } else {
            bind_slot(slot, R, &Pc);
            R.ticket = ++p->ticket; R.pdl = overlap_ok ? 1 : 0;
            Pc.ticket = R.ticket;
            wait_for_slot(slot, R);
            CK(launch_resolve(R, stream));
            g_launches++;
            overlap_ok = true;                              // the kernels behind it may overlap IT
        }
        p->cur_slot = slot;
        p->ahead_valid = false;
        {   // speculate on the next call: same everything, first_index advanced by the stride seen so far
            uint64_t stride = (uint64_t)batch;
            faa_policy::AheadKey base = key; base.first_index = 0;
            faa_policy::AheadKey lastb = p->last_key; lastb.first_index = 0;
            if (p->have_last && memcmp(&base, &lastb, sizeof base) == 0 && rng->first_index > p->last_key.first_index)
                stride = rng->first_index - p->last_key.first_index;
            p->last_key = key; p->have_last = true;
            ResolveParams R2 = R;
            R2.rng.first_index = rng->first_index + stride;
            bind_slot(slot ^ 1, R2, nullptr);
            R2.ticket = ++p->ticket; R2.pdl = overlap_ok ? 1 : 0;
            // (its slot's last readers - the step before this one - copied their programs before they let any
            //  later kernel of the stream start, so the resolve kernel may overwrite the slot as soon as it runs;
            //  persistent readers release their dependents at once and are waited for through the slot's counter)
            wait_for_slot(slot ^ 1, R2);
            CK(launch_resolve(R2, stream));
            g_launches++;
            p->ahead_key = key; p->ahead_key.first_index = rng->first_index + stride;
            p->ahead_slot = slot ^ 1; p->ahead_valid = true; p->ahead_ticket = R2.ticket;
        }
        if (persist) {
            if (!p->sm_count) CK(cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, p->device));
            Pc.done = done_word(slot);
            if (P.scratch) Pc.scratch = P.scratch + (size_t)slot * scratch_half;
        }
        AugParams Pm = Pc;                                  // the mid kernel: its own (taller) bands in bands / geo[0]
        if (use_mid) set_mid_geometry(Pm);
        if (persist) {
            // one resident wave each (launch bounds: light CTAs / SM, 2 mid CTAs / SM)
            static const int rows_l = [] { const char* e = getenv("FAA_ROWS_LIGHT"); return e ? atoi(e) : 0; }();
            static const int rows_m = [] { const char* e = getenv("FAA_ROWS_MID"); return e ? atoi(e) : 0; }();
            const int lb = P.geo[1].bands > 0 ? P.geo[1].bands : 1;
            Pc.grid_y = rows_l > 0 ? rows_l : (p->sm_count * resident_ctas_per_sm(1)) / lb;
            // (mid rows: ONE CTA per SM measured best - 58.1 us vs 58.9 us with both slots - the light CTAs that follow
            //  share the SM with it from the start; profiles/r02_schedules.txt)
            Pm.grid_y = rows_m > 0 ? rows_m : p->sm_count / (Pm.bands > 0 ? Pm.bands : 1);
            if (Pc.grid_y < 1) Pc.grid_y = 1;
            if (Pm.grid_y < 1) Pm.grid_y = 1;
        }
        const int order3[3] = {chain_mode == 2 ? 1 : 0, 2, chain_mode == 2 ? 0 : 1};   // default: cluster, mid, light
        for (int k = 0; k < 3; ++k) {
            const int which = order3[k];
            if (which != 0 && !use_split) continue;          // one pixel kernel
            if (which == 2) { if (use_mid) { CK(launch_augment(Pm, tail->out_dtype, use_tab, 2, stream)); g_launches++; if (persist) p->done_target[slot] += augment_cta_count(Pm, 2); } }
            else if (which == 0 && no_heavy) continue;
            else {
                AugParams Pk = Pc;
                if (which == 0) Pk.grid_y = 0;              // the cluster kernel keeps one cluster per entry
                CK(launch_augment(Pk, tail->out_dtype, use_tab, which, stream)); g_launches++;
                if (persist) p->done_target[slot] += augment_cta_count(Pk, which);
            }
        }
        p->chain_live = true; p->chain_stream = stream;
        p->prev_in[0] = in0; p->prev_in[1] = in1; p->prev_out[0] = out0; p->prev_out[1] = out1;
        return FAA_OK;
    }
    p->chain_live = false;
    if (hit) {
        slot = p->ahead_slot;
        CK(cudaStreamWaitEvent(stream, p->ev_ahead, 0));
        P.pdl = 0;                                          // no resolve kernel right in front of the pixel kernel
        bind_slot(slot, R, &P);
    } else {
        bind_slot(slot, R, &P);
        CK(launch_resolve(R, stream));
        g_launches++;
    }
    p->cur_slot = slot;
    p->ahead_valid = false;
    if (P.n_heavy || spec_ok) {
        if (!p->light_stream) {
            {
                int lo = 0, hi = 0;
                CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));       // hi = numerically lowest = greatest priority
                CK(cudaStreamCreateWithPriority(&p->light_stream, cudaStreamNonBlocking, hi));
            }
            {
                int lo = 0, hi = 0;
                CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
                CK(cudaStreamCreateWithPriority(&p->ahead_stream, cudaStreamNonBlocking, hi));   // one block: get a slot promptly
            }
            {
                int lo = 0, hi = 0;
                CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
                CK(cudaStreamCreateWithPriority(&p->mid_stream, cudaStreamNonBlocking, hi));
            }
            CK(cudaEventCreateWithFlags(&p->ev_mid, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&p->ev_res, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&p->ev_light, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&p->ev_ahead, cudaEventDisableTiming));
        }
        CK(cudaEventRecord(p->ev_res, stream));               // this batch's programs are ready
    }
    if (spec_ok) {
        // speculate on the next call: same everything, first_index advanced by the stride seen so far
        uint64_t stride = (uint64_t)batch;
        faa_policy::AheadKey base = key; base.first_index = 0;
        faa_policy::AheadKey lastb = p->last_key; lastb.first_index = 0;
        if (p->have_last && memcmp(&base, &lastb, sizeof base) == 0 && rng->first_index > p->last_key.first_index)
            stride = rng->first_index - p->last_key.first_index;
        p->last_key = key; p->have_last = true;
        ResolveParams R2 = R;
        R2.rng.first_index = rng->first_index + stride;
        bind_slot(slot ^ 1, R2, nullptr);
        CK(cudaStreamWaitEvent(p->ahead_stream, p->ev_res, 0));      // the other slot's last readers are done
        CK(launch_resolve(R2, p->ahead_stream));
        CK(cudaEventRecord(p->ev_ahead, p->ahead_stream));
        g_launches++;
        p->ahead_key = key; p->ahead_key.first_index = rng->first_index + stride;
        p->ahead_slot = slot ^ 1; p->ahead_valid = true;
    }
    // launch 2: pixels
    if (P.n_heavy) {
        // Two pixel kernels, concurrently: the light streaming kernel goes first on the caller's
        // stream and fills the machine; the cluster kernel runs on a HIGH-PRIORITY side stream, so its
        // clusters take the CTA slots as they free up (heavy images finish early, light work fills gaps).
        static const bool prio_off = [] { const char* e = getenv("FAA_PRIO"); return e && e[0] == '0'; }();
        if (prio_off) {
            CK(cudaStreamWaitEvent(p->light_stream, p->ev_res, 0));
            CK(launch_augment(P, tail->out_dtype, use_tab, 0, stream));
            CK(launch_augment(P, tail->out_dtype, use_tab, 1, p->light_stream));
            if (use_mid) { AugParams Pm = P; Pm.pdl = 0; set_mid_geometry(Pm); CK(launch_augment(Pm, tail->out_dtype, use_tab, 2, p->light_stream)); g_launches++; }
            CK(cudaEventRecord(p->ev_light, p->light_stream));
        } else {
            AugParams Ph = P; Ph.pdl = 0;                           // not behind the resolve kernel in its stream
            CK(cudaStreamWaitEvent(p->light_stream, p->ev_res, 0));
            static const bool mid_same = [] { const char* e = getenv("FAA_MID_STREAM"); return e && e[0] == '0'; }();
            static const int order_knob = [] { const char* e = getenv("FAA_ORDER"); return e ? atoi(e) : 0; }();
            if (use_mid && !mid_same) CK(cudaStreamWaitEvent(p->mid_stream, p->ev_res, 0));
            // the streaming kernel goes FIRST: it fills the machine at once; the priority streams' clusters then take
            // the slots its CTAs free (launched first, the thousands of exiting CTAs of the cluster kernels would hold
            // up the work distributor: measured +10 us per step)
            if (order_knob == 0) CK(launch_augment(P, tail->out_dtype, use_tab, 1, stream));
            if (!no_heavy) CK(launch_augment(Ph, tail->out_dtype, use_tab, 0, p->light_stream)); else g_launches--;
            if (order_knob == 1) CK(launch_augment(P, tail->out_dtype, use_tab, 1, stream));
            if (use_mid) {                                                               // statistics / Sharpness clusters: third stream
                AugParams Pm = Ph; set_mid_geometry(Pm);
                CK(launch_augment(Pm, tail->out_dtype, use_tab, 2, mid_same ? p->light_stream : p->mid_stream)); g_launches++;
                if (!mid_same) CK(cudaEventRecord(p->ev_mid, p->mid_stream));
            }
            if (order_knob == 2) CK(launch_augment(P, tail->out_dtype, use_tab, 1, stream));
            CK(cudaEventRecord(p->ev_light, p->light_stream));
            if (use_mid && !mid_same) CK(cudaStreamWaitEvent(stream, p->ev_mid, 0));
        }
        CK(cudaStreamWaitEvent(stream, p->ev_light, 0));
        g_launches += 2;
    } else {
        CK(launch_augment(P, tail->out_dtype, use_tab, 0, stream));
        g_launches++;
    }
    return FAA_OK;
}

int faa_augment(faa_policy_t* p, const uint8_t* d_in, void* d_out, int batch, int h, int w, const faa_tail_t* tail,
                const faa_sample_t* d_samples, const faa_box_t* d_boxes, const faa_rng_t* rng, int op_base,
                void* stream) {
    if (!p) return fail(FAA_ERR_VALUE, "null policy");
    // intermediate launch of a chained policy = not the last 2-op window
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    int apply_tail = (op_base + FAA_MAX_FUSED_OPS >= p->n_op) ? 1 : 0;
    if (!apply_tail && tail && (tail->out_dtype != FAA_U8_HWC || tail->out_h != h || tail->out_w != w))
        return fail(FAA_ERR_VALUE, "intermediate launches of a chained policy must write uint8 HWC at the input size");
    return augment_common(p, d_in, batch, 0, d_out, batch, h, w, tail, d_samples, d_boxes, rng, op_base, nullptr,
                          1.0f, 0.0f, apply_tail, p->n_op <= FAA_MAX_FUSED_OPS, stream);
}

int faa_policy_set_overlap(faa_policy_t* p, int on) {
    if (!p) return fail(FAA_ERR_VALUE, "null policy");
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    p->overlap_calls = on != 0;
    return FAA_OK;
}

int faa_augment_many(faa_policy_t* p, int n_steps, const uint8_t* const* d_in, void* const* d_out, int batch, int h, int w,
                     const faa_tail_t* tail, const faa_rng_t* rng, uint64_t index_stride, void* stream) {
    if (!p || !rng || !d_in || !d_out) return fail(FAA_ERR_VALUE, "null argument");
    if (n_steps < 0) return fail(FAA_ERR_VALUE, "bad step count");
    if (p->n_op > FAA_MAX_FUSED_OPS) return fail(FAA_ERR_UNSUPPORTED, "multi-step launches support policies of at most 2 ops");
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    faa_rng_t r = *rng;
    const bool saved = p->overlap_calls;
    int rc = FAA_OK;
    for (int k = 0; k < n_steps && rc == FAA_OK; ++k) {
        // every input exists before this call: steps 2.. may overlap their predecessor; step 1 follows whatever the caller
        // issued before (stream order) unless the caller made the promise for whole calls too
        p->overlap_calls = k > 0 ? true : saved;
        rc = augment_common(p, d_in[k], batch, 0, d_out[k], batch, h, w, tail, nullptr, nullptr, &r, 0, nullptr,
                            1.0f, 0.0f, 1, true, stream);
        r.first_index += index_stride;
    }
    p->overlap_calls = saved;
    return rc;
}

int faa_augment_tta(faa_policy_t* p, const uint8_t* d_in, void* d_out, int batch, int replicas, int h, int w,
                    const faa_tail_t* tail, const faa_rng_t* rng, void* stream) {
    if (!p || !rng) return fail(FAA_ERR_VALUE, "null argument");
    if (p->n_op > FAA_MAX_FUSED_OPS) return fail(FAA_ERR_UNSUPPORTED, "replicated launches support policies of at most 2 ops");
    if (batch < 0 || replicas < 1) return fail(FAA_ERR_VALUE, "bad batch / replicas");
    if ((long long)batch * replicas > 65535) return fail(FAA_ERR_UNSUPPORTED, "batch * replicas must be <= 65535");
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    // one launch over batch * replicas schedule entries; entry v = r * batch + i reads image i and draws the decisions of
    // global sample first_index + v: replica r equals a plain launch with first_index + r * batch
    return augment_common(p, d_in, batch * replicas, 0, d_out, batch * replicas, h, w, tail, nullptr, nullptr, rng, 0, nullptr,
                          1.0f, 0.0f, 1, true, stream, replicas > 1 ? batch : 0);
}

int faa_augment_mixup(faa_policy_t* p, const uint8_t* d_in_all, int n_all, int first, void* d_out, int batch, int h,
                      int w, const faa_tail_t* tail, const faa_sample_t* d_samples_all, const faa_box_t* d_boxes_all,
                      const faa_rng_t* rng, const int32_t* d_partner, float lam, float one_minus_lam, void* stream) {
    if (!p) return fail(FAA_ERR_VALUE, "null policy");
    if (p->n_op > FAA_MAX_FUSED_OPS) return fail(FAA_ERR_UNSUPPORTED, "fused mixup supports policies of at most 2 ops");
    if (!(lam >= 0.0f && lam <= 1.0f)) return fail(FAA_ERR_MAGNITUDE, "lam must be in [0, 1]");   // aug_mixup.py:20
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    return augment_common(p, d_in_all, n_all, first, d_out, batch, h, w, tail, d_samples_all, d_boxes_all, rng, 0,
                          d_partner, lam, one_minus_lam, 1, false, stream);
}

int faa_policy_set_lighting(faa_policy_t* p, const float* d_rgb, int n) {
    if (!p) return fail(FAA_ERR_VALUE, "null policy");
    if (d_rgb && n <= 0) return fail(FAA_ERR_VALUE, "n must be positive");
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    p->lighting_rgb = d_rgb; p->lighting_n = d_rgb ? n : 0;
    return FAA_OK;
}

int faa_color_jitter(const uint8_t* d_in, uint8_t* d_out, int batch, int h, int w, const faa_jitter_t* d_recs, void* stream) {
    if ((!d_in || !d_out || !d_recs) && batch > 0) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0) return fail(FAA_ERR_VALUE, "negative batch");
    if (int e = check_shape(h, w)) return e;
    if (int e = ensure_device()) return e;
    static_assert(sizeof(faa_jitter_t) == 16, "jitter record is 16 bytes");
    CK(launch_color_jitter(d_in, d_out, d_recs, batch, h, w, (cudaStream_t)stream));
    if (batch > 0) g_launches++;
    return FAA_OK;
}

int faa_mix_u8(faa_policy_t* p, const uint8_t* d_a, const uint8_t* d_b, const int32_t* d_partner, const int16_t* d_zero_box_a,
               const int16_t* d_zero_box_b, void* d_out, int batch, int h, int w, const faa_tail_t* tail, float lam,
               float one_minus_lam, void* stream) {
    if (!p || ((!d_a || !d_b || !d_partner || !d_out) && batch > 0)) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0) return fail(FAA_ERR_VALUE, "negative batch");
    if (int e = check_shape(h, w)) return e;
    if (int e = check_tail(tail)) return e;
    if (tail->out_dtype == FAA_U8_HWC) return fail(FAA_ERR_UNSUPPORTED, "mixup needs a float output");
    if (tail->out_h != h || tail->out_w != w) return fail(FAA_ERR_VALUE, "the augmented images already have the output size");
    if ((w & 3) || ((uintptr_t)d_a & 3) || ((uintptr_t)d_b & 3) || ((uintptr_t)d_out & 15))
        return fail(FAA_ERR_UNSUPPORTED, "faa_mix_u8 needs W % 4 == 0 and aligned buffers");
    if (!(lam >= 0.0f && lam <= 1.0f)) return fail(FAA_ERR_MAGNITUDE, "lam must be in [0, 1]");   // aug_mixup.py:20
    if (int e = ensure_device()) return e;
    if (batch == 0) return FAA_OK;
    if (int e = bind_device(p)) return e;
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    AugParams dummy; bool tab = false;
    if (int e = normalisation(p, tail, dummy, tab, (cudaStream_t)stream)) return e;
    CK(launch_mix_u8(d_a, d_b, d_partner, d_zero_box_a, d_zero_box_b, p->d_norm, d_out, batch, h, w, tail->out_dtype, lam,
                     one_minus_lam, (cudaStream_t)stream));
    g_launches++;
    return FAA_OK;
}

int faa_enable_peer_access(int peer_device) {
    if (int e = ensure_device()) return e;
    int dev = -1, can = 0;
    CK(cudaGetDevice(&dev));
    if (peer_device == dev) return FAA_OK;
    CK(cudaDeviceCanAccessPeer(&can, dev, peer_device));
    if (!can) return fail(FAA_ERR_UNSUPPORTED, "device " + std::to_string(dev) + " cannot access the memory of device " + std::to_string(peer_device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return FAA_OK; }
    CK(e);
    return FAA_OK;
}

// ---- buffers other processes of the node can map (CUDA IPC): the Mixup partner pool -------------------------------
int faa_peer_alloc(size_t bytes, void** d_ptr, unsigned char* handle64) {
    if (!d_ptr || !handle64 || bytes == 0) return fail(FAA_ERR_VALUE, "bad argument");
    if (int e = ensure_device()) return e;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void* p = nullptr;
    CK(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    if (cudaError_t e = cudaIpcGetMemHandle(&h, p)) { cudaFree(p); CK(e); }
    CK(cudaMemset(p, 0, bytes));
    memcpy(handle64, &h, 64);
    *d_ptr = p;
    return FAA_OK;
}

int faa_peer_open(const unsigned char* handle64, void** d_ptr) {
    if (!d_ptr || !handle64) return fail(FAA_ERR_VALUE, "bad argument");
    if (int e = ensure_device()) return e;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    // opened under the CURRENT device: lazy peer access lets this device's kernels dereference the mapping
    CK(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return FAA_OK;
}

int faa_peer_close(void* d_ptr) { if (d_ptr) CK(cudaIpcCloseMemHandle(d_ptr)); return FAA_OK; }
int faa_peer_free(void* d_ptr) { if (d_ptr) CK(cudaFree(d_ptr)); return FAA_OK; }

int faa_mix_u8_peer(faa_policy_t* p, const uint8_t* d_a, const uint8_t* const* d_partner_ptrs, const int16_t* d_zero_box_a,
                    const int16_t* d_zero_box_b, void* d_out, int batch, int h, int w, const faa_tail_t* tail, float lam,
                    float one_minus_lam, void* stream) {
    if (!p || ((!d_a || !d_partner_ptrs || !d_out) && batch > 0)) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0) return fail(FAA_ERR_VALUE, "negative batch");
    if (int e = check_shape(h, w)) return e;
    if (int e = check_tail(tail)) return e;
    if (tail->out_dtype == FAA_U8_HWC) return fail(FAA_ERR_UNSUPPORTED, "mixup needs a float output");
    if (tail->out_h != h || tail->out_w != w) return fail(FAA_ERR_VALUE, "the augmented images already have the output size");
    if ((w & 3) || ((uintptr_t)d_a & 3) || ((uintptr_t)d_out & 15) || ((uintptr_t)d_partner_ptrs & 7))
        return fail(FAA_ERR_UNSUPPORTED, "faa_mix_u8_peer needs W % 4 == 0 and aligned buffers");
    if (!(lam >= 0.0f && lam <= 1.0f)) return fail(FAA_ERR_MAGNITUDE, "lam must be in [0, 1]");   // aug_mixup.py:20
    if (int e = ensure_device()) return e;
    if (batch == 0) return FAA_OK;
    if (int e = bind_device(p)) return e;
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    AugParams dummy; bool tab = false;
    if (int e = normalisation(p, tail, dummy, tab, (cudaStream_t)stream)) return e;
    CK(launch_mix_u8(d_a, nullptr, nullptr, d_zero_box_a, d_zero_box_b, p->d_norm, d_out, batch, h, w, tail->out_dtype, lam,
                     one_minus_lam, (cudaStream_t)stream, d_partner_ptrs));
    g_launches++;
    return FAA_OK;
}

int faa_mixup(const void* d_data, void* d_out, const int64_t* d_perm, int batch, int64_t n_per_sample, int dtype,
              float lam, float one_minus_lam, void* stream) {
    if ((!d_data || !d_out || !d_perm) && batch > 0) return fail(FAA_ERR_VALUE, "null argument");
    if (batch < 0 || n_per_sample < 0) return fail(FAA_ERR_VALUE, "negative size");
    if (dtype < 0 || dtype > FAA_F32) return fail(FAA_ERR_VALUE, "bad dtype");
    if (int e = ensure_device()) return e;
    CK(launch_mixup(d_data, d_out, d_perm, batch, n_per_sample, dtype, lam, one_minus_lam, (cudaStream_t)stream));
    if (batch > 0 && n_per_sample > 0) g_launches++;
    return FAA_OK;
}

// ------------------------------------------------------------- host buffers --
static int grow_dev(void** ptr, size_t* have, size_t need) {
    if (*have >= need) return FAA_OK;
    if (*ptr) { CK(cudaFree(*ptr)); *ptr = nullptr; *have = 0; }
    CK(cudaMalloc(ptr, need));
    *have = need;
    return FAA_OK;
}
static int grow_pinned(void** ptr, size_t* have, size_t need) {
    if (*have >= need) return FAA_OK;
    if (*ptr) { CK(cudaFreeHost(*ptr)); *ptr = nullptr; *have = 0; }
    CK(cudaMallocHost(ptr, need));
    *have = need;
    return FAA_OK;
}
static bool is_pinned(const void* ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

int faa_augment_host(faa_policy_t* p, const uint8_t* h_in, void* h_out, void* d_out_keep, int batch, int h, int w,
                     const faa_tail_t* tail, const faa_rng_t* rng, void* stream_v) {
    if (!p || !h_in || !rng) return fail(FAA_ERR_VALUE, "null argument");
    if (p->n_op > FAA_MAX_FUSED_OPS) return fail(FAA_ERR_UNSUPPORTED, "host-buffer entry supports policies of at most 2 ops");
    if (int e = check_shape(h, w)) return e;
    if (int e = check_tail(tail)) return e;
    if (int e = ensure_device()) return e;
    if (batch <= 0) return FAA_OK;
    if (int e = bind_device(p)) return e;
    cudaStream_t stream = (cudaStream_t)stream_v;
    std::lock_guard<std::mutex> call_lk(p->call_mu);
    // The policy owns the device input buffer and the pinned stages: the previous call's asynchronous copies must
    // have finished before any of them is rewritten (a pageable source is memcpy'd into the stage right below)
    if (p->host_in_flight) { CK(cudaEventSynchronize(p->ev_host_done)); p->host_in_flight = false; }
    if (!p->ev_host_done) CK(cudaEventCreateWithFlags(&p->ev_host_done, cudaEventDisableTiming));
    const size_t in_img = (size_t)h * w * 3;
    const size_t out_img = (size_t)tail->out_h * tail->out_w * 3 * out_elem_size(tail->out_dtype);
    if (int e = grow_dev(&p->d_in, &p->d_in_bytes, in_img * batch)) return e;
    void* d_out = d_out_keep;
    if (!d_out) { if (int e = grow_dev(&p->d_out, &p->d_out_bytes, out_img * batch)) return e; d_out = p->d_out; }
    for (int i = 0; i < 2; ++i) {
        if (!p->side[i]) CK(cudaStreamCreateWithFlags(&p->side[i], cudaStreamNonBlocking));
        if (!p->ev_join[i]) CK(cudaEventCreateWithFlags(&p->ev_join[i], cudaEventDisableTiming));
    }
    if (!p->ev_fork) CK(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));

    // pageable buffers are staged through pinned memory (synchronous host copies)
    const bool in_pinned = is_pinned(h_in);
    const bool out_pinned = !h_out || is_pinned(h_out);
    const uint8_t* src = h_in;
    if (!in_pinned) {
        if (int e = grow_pinned(&p->h_in_stage, &p->h_in_bytes, in_img * batch)) return e;
        memcpy(p->h_in_stage, h_in, in_img * batch);
        src = (const uint8_t*)p->h_in_stage;
    }
    void* dst = h_out;
    if (h_out && !out_pinned) {
        if (int e = grow_pinned(&p->h_out_stage, &p->h_out_bytes, out_img * batch)) return e;
        dst = p->h_out_stage;
    }

    // tables the side streams will read are uploaded on `stream` before the fork
    if (tail->out_dtype != FAA_U8_HWC) {
        AugParams dummy; bool tab = false;
        if (int e = normalisation(p, tail, dummy, tab, stream)) return e;
    }
    {
        const OpRec* d_ops = nullptr;
        if (int e = device_table(p, h, w, true, &d_ops)) return e;
    }
    // chunked pipeline on two side streams: H2D(c+1) overlaps kernel(c) and D2H(c)
    int chunks = batch >= 64 ? 8 : (batch >= 8 ? 2 : 1);
    CK(cudaEventRecord(p->ev_fork, stream));
    CK(cudaStreamWaitEvent(p->side[0], p->ev_fork, 0));
    CK(cudaStreamWaitEvent(p->side[1], p->ev_fork, 0));
    for (int c = 0; c < chunks; ++c) {
        int b0 = (int)((long long)batch * c / chunks), b1 = (int)((long long)batch * (c + 1) / chunks);
        if (b1 <= b0) continue;
        cudaStream_t s = p->side[c & 1];
        CK(cudaMemcpyAsync((uint8_t*)p->d_in + in_img * b0, src + in_img * b0, in_img * (b1 - b0), cudaMemcpyHostToDevice, s));
        if (int e = augment_common(p, (const uint8_t*)p->d_in, batch, b0, (uint8_t*)d_out + out_img * b0, b1 - b0, h, w,
                                   tail, nullptr, nullptr, rng, 0, nullptr, 1.0f, 0.0f, 1, false, s)) return e;
        if (dst) CK(cudaMemcpyAsync((uint8_t*)dst + out_img * b0, (uint8_t*)d_out + out_img * b0, out_img * (b1 - b0), cudaMemcpyDeviceToHost, s));
    }
    for (int i = 0; i < 2; ++i) {
        CK(cudaEventRecord(p->ev_join[i], p->side[i]));
        CK(cudaStreamWaitEvent(stream, p->ev_join[i], 0));
    }
    CK(cudaEventRecord(p->ev_host_done, stream));
    p->host_in_flight = true;
    if (h_out && !out_pinned) {
        CK(cudaStreamSynchronize(stream));
        memcpy(h_out, p->h_out_stage, out_img * batch);
    }
    return FAA_OK;
}

}  // extern "C"
