// oracle/ref_record.cpp -- TEST INFRASTRUCTURE ONLY: a preload library for the oracle-served drop-in harness
// (_ref/ref_backend_orc).  It interposes the orc_ba_* entry points the product shim calls, appends every bundle-adjustment
// problem the reference's own code hands to the solver -- parameter blocks, factor arrays, losses, options -- and what the
// oracle's solve returned to the file named by LVB_RECORD, then forwards each call.  tests/golden/make_ref_golden.py turns
// the log into tests/golden/ref_backend.npz, so the comparison with those problems runs where the reference tree is absent.
//
// Log: a sequence of records, each an int32 tag followed by its payload (native byte order).
#include <dlfcn.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../include/lvio_b200.h"

namespace {
enum Tag : int32_t { CREATE = 1, CAMERAS, POSES, VEC3, INV_DEPTHS, FACTORS, LOSS, SOLVE };
const int kConst[LVB_NUM_KINDS] = {5, 6, 5, 469, 8, 9};
const int kIdx[LVB_NUM_KINDS] = {3, 1, 1, 8, 2, 1};
int g_n[3];                                                     // poses, vec3, inverse depths of the open problem

FILE* out() {
    static FILE* f = [] {
        const char* p = std::getenv("LVB_RECORD");
        FILE* h = p ? std::fopen(p, "wb") : nullptr;
        if (!h) { std::fprintf(stderr, "ref_record: LVB_RECORD is not a writable path\n"); std::abort(); }
        return h;
    }();
    return f;
}
void put(const void* p, size_t bytes) { if (bytes && std::fwrite(p, 1, bytes, out()) != bytes) std::abort(); }
void put_i(int32_t v) { put(&v, sizeof(v)); }
void put_d(double v) { put(&v, sizeof(v)); }
template <class F> F next(const char* name) {
    void* f = dlsym(RTLD_NEXT, name);
    if (!f) { std::fprintf(stderr, "ref_record: %s not found\n", name); std::abort(); }
    return reinterpret_cast<F>(f);
}
void blocks(Tag tag, int slot, int n, int width, const double* v, const uint8_t* is_const) {
    g_n[slot] = n;
    put_i(tag); put_i(n); put(v, sizeof(double) * n * width);
    put_i(is_const ? 1 : 0);
    if (is_const) put(is_const, n);
}
}  // namespace

extern "C" {
int orc_ba_create(lvb_ctx* ctx, lvb_ba** o) {
    put_i(CREATE);
    return next<int (*)(lvb_ctx*, lvb_ba**)>("orc_ba_create")(ctx, o);
}
int orc_ba_set_cameras(lvb_ba* ba, const double cam[22]) {
    put_i(CAMERAS); put(cam, 22 * sizeof(double));
    return next<int (*)(lvb_ba*, const double*)>("orc_ba_set_cameras")(ba, cam);
}
int orc_ba_set_poses(lvb_ba* ba, int n, const double* v, const uint8_t* c) {
    blocks(POSES, 0, n, 7, v, c);
    return next<int (*)(lvb_ba*, int, const double*, const uint8_t*)>("orc_ba_set_poses")(ba, n, v, c);
}
int orc_ba_set_vec3(lvb_ba* ba, int n, const double* v, const uint8_t* c) {
    blocks(VEC3, 1, n, 3, v, c);
    return next<int (*)(lvb_ba*, int, const double*, const uint8_t*)>("orc_ba_set_vec3")(ba, n, v, c);
}
int orc_ba_set_inv_depths(lvb_ba* ba, int n, const double* v, const uint8_t* c) {
    blocks(INV_DEPTHS, 2, n, 1, v, c);
    return next<int (*)(lvb_ba*, int, const double*, const uint8_t*)>("orc_ba_set_inv_depths")(ba, n, v, c);
}
int orc_ba_add_factors(lvb_ba* ba, int kind, int n, const double* consts, const int32_t* idx) {
    if (kind < 0 || kind >= LVB_NUM_KINDS) std::abort();
    put_i(FACTORS); put_i(kind); put_i(n);
    put(consts, sizeof(double) * n * kConst[kind]); put(idx, sizeof(int32_t) * n * kIdx[kind]);
    return next<int (*)(lvb_ba*, int, int, const double*, const int32_t*)>("orc_ba_add_factors")(ba, kind, n, consts, idx);
}
int orc_ba_set_loss(lvb_ba* ba, int kind, double a) {
    put_i(LOSS); put_i(kind); put_d(a);
    return next<int (*)(lvb_ba*, int, double)>("orc_ba_set_loss")(ba, kind, a);
}
// options as 10 doubles, then the summary (5 doubles) and the solved blocks the oracle returns
int orc_ba_solve(lvb_ba* ba, const lvb_solve_options* o, lvb_solve_summary* s) {
    const int rc = next<int (*)(lvb_ba*, const lvb_solve_options*, lvb_solve_summary*)>("orc_ba_solve")(ba, o, s);
    put_i(SOLVE);
    const double opt[10] = {(double)o->max_num_iterations, o->max_solver_time_in_seconds, o->function_tolerance, o->gradient_tolerance,
                            o->parameter_tolerance, o->initial_trust_region_radius, (double)o->jacobi_scaling, (double)o->linear_solver_type,
                            (double)o->num_threads, (double)o->schur_mode};
    put(opt, sizeof(opt));
    const double sum[6] = {(double)rc, s->initial_cost, s->final_cost, (double)s->num_iterations, (double)s->num_successful_steps, (double)s->termination_type};
    put(sum, sizeof(sum));
    const int w[3] = {7, 3, 1};
    const char* get[3] = {"orc_ba_get_poses", "orc_ba_get_vec3", "orc_ba_get_inv_depths"};
    for (int k = 0; k < 3; ++k) {
        double* v = (double*)std::calloc((size_t)g_n[k] * w[k] + 1, sizeof(double));
        if (g_n[k] && next<int (*)(lvb_ba*, double*)>(get[k])(ba, v) != LVB_OK) std::abort();
        put(v, sizeof(double) * g_n[k] * w[k]);
        std::free(v);
    }
    std::fflush(out());
    return rc;
}
}
