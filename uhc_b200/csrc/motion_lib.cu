// motion_lib.cu -- expert tables built on the device from raw SMPL pose sequences (include/uhc_motion.h): uhc_load_clips_smpl,
// uhc_get_clip_frames.
//
// Replaces the host path of a dataset load (make_expert per clip in numpy fp64, pack_expert into [frames][576] doubles, a float conversion
// loop and the upload in uhc_load_clips): the upload is the input rows (72 or 156 doubles + 3 per frame), one thread per frame computes its
// record with the math of motion_fk.h and writes it into a new table, which replaces the engine's table only once it is complete and valid.
// Built without FMA contraction (uhc_b200/build.py), so the fp64 records match the host motion library to the last bits except where the
// libm and CUDA transcendentals differ.
#include <cuda_runtime.h>
#include <math.h>
#include <string>
#include <vector>
#include "../../include/uhc_b200.h"
#include "../../include/uhc_motion.h"
#include "clip_table.h"
#include "eval_internal.h"
#include "motion_fk.h"

#define CKM(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { uhc_engine_set_error((std::string(#x) + ": " + cudaGetErrorString(e_)).c_str()); return -1; } } while (0)

namespace {

constexpr int THREADS = 128;

// one thread per frame: the clip by binary search over clip_adr, then the frame's record; a non-finite value in the frame's input row sets *bad
template <class Out>
__global__ void __launch_bounds__(THREADS)
k_expert_frames(const double *__restrict__ pose, int pose_dim, const double *__restrict__ trans, const int *__restrict__ clip_adr, int nclips,
                const int *__restrict__ clip_model, const double *__restrict__ off_ipos, const int *__restrict__ topo, int total, Out *__restrict__ out,
                int *__restrict__ bad) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total) return;
    int lo = 0, hi = nclips - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (clip_adr[mid] <= f) lo = mid; else hi = mid - 1; }
    const int base = clip_adr[lo];
    bool finite = true;
    for (int k = 0; k < pose_dim; k++) finite &= isfinite(pose[(size_t)f * pose_dim + k]);
    if (trans) for (int k = 0; k < 3; k++) finite &= isfinite(trans[(size_t)f * 3 + k]);
    if (!finite) *bad = 1;
    const uhc_motion::Kin kin{off_ipos + (size_t)(clip_model ? clip_model[lo] : 0) * uhc_motion::NB * 6, topo, topo + uhc_motion::NB};
    uhc_motion::expert_frame<Out>(pose + (size_t)base * pose_dim, pose_dim, trans ? trans + (size_t)base * 3 : nullptr, f - base, kin,
                                  out + (size_t)f * uhc_motion::REC);
}

// device buffers of one call, freed on every return unless released into the engine
struct Scratch {
    std::vector<void *> p;
    template <class T> cudaError_t alloc(T **d, size_t n) { cudaError_t r = cudaMalloc((void **)d, n * sizeof(T)); if (r == cudaSuccess) p.push_back(*d); return r; }
    void release(const void *d) { for (auto &q : p) if (q == d) q = nullptr; }
    ~Scratch() { for (void *q : p) if (q) cudaFree(q); }
};

int fail(const char *msg) { uhc_engine_set_error(msg); return -2; }

template <class Real>
int build_table(UhcEngine *e, int nclips, const int *clip_len, int pose_dim, const double *pose_host, const double *trans_host,
                const double *shape_host, const int *clip_model_host, const EngineKin &kin, size_t total) {
    Scratch s;
    double *d_pose, *d_trans = nullptr, *d_kin;
    int *d_int;
    Real *d_out, *d_shape;
    const size_t nkin = (size_t)kin.nshape * uhc_motion::NB * 6;
    // ints: clip_adr [C + 1], clip_model [C], parent [24], ee [5], bad flag
    std::vector<int> ints((size_t)2 * nclips + 1 + uhc_motion::NB + 5 + 1, 0);
    for (int c = 0; c < nclips; c++) { ints[c + 1] = ints[c] + clip_len[c]; ints[nclips + 1 + c] = clip_model_host ? clip_model_host[c] : 0; }
    for (int b = 0; b < uhc_motion::NB; b++) ints[2 * nclips + 1 + b] = kin.parent[b];
    for (int k = 0; k < 5; k++) ints[2 * nclips + 1 + uhc_motion::NB + k] = kin.ee[k];
    CKM(s.alloc(&d_pose, total * pose_dim));
    CKM(cudaMemcpy(d_pose, pose_host, total * pose_dim * sizeof(double), cudaMemcpyHostToDevice));
    if (trans_host) { CKM(s.alloc(&d_trans, total * 3)); CKM(cudaMemcpy(d_trans, trans_host, total * 3 * sizeof(double), cudaMemcpyHostToDevice)); }
    CKM(s.alloc(&d_kin, nkin)); CKM(cudaMemcpy(d_kin, kin.off_ipos, nkin * sizeof(double), cudaMemcpyHostToDevice));
    CKM(s.alloc(&d_int, ints.size())); CKM(cudaMemcpy(d_int, ints.data(), ints.size() * sizeof(int), cudaMemcpyHostToDevice));
    CKM(s.alloc(&d_out, total * uhc_motion::REC));
    std::vector<Real> shp((size_t)nclips * 17);
    for (size_t i = 0; i < shp.size(); i++) shp[i] = (Real)shape_host[i];
    CKM(s.alloc(&d_shape, shp.size())); CKM(cudaMemcpy(d_shape, shp.data(), shp.size() * sizeof(Real), cudaMemcpyHostToDevice));
    int *d_bad = d_int + ints.size() - 1;
    k_expert_frames<Real><<<(unsigned)((total + THREADS - 1) / THREADS), THREADS>>>(d_pose, pose_dim, d_trans, d_int, nclips,
                                                                                  clip_model_host ? d_int + nclips + 1 : nullptr, d_kin,
                                                                                  d_int + 2 * nclips + 1, (int)total, d_out, d_bad);
    CKM(cudaGetLastError());
    int bad = 0;
    CKM(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) return fail("uhc_load_clips_smpl: non-finite pose or trans value");
    const int rc = uhc_engine_install_clips(e, nclips, clip_len, d_out, d_shape);
    if (rc) return rc;
    s.release(d_out); s.release(d_shape);
    return clip_model_host ? uhc_set_clip_models(e, nclips, clip_model_host) : 0;
}

}  // namespace

extern "C" {

int uhc_load_clips_smpl(UhcEngine *e, int nclips, const int *clip_len, int pose_dim, const double *pose_host, const double *trans_host,
                        const double *shape_host, const int *clip_model_host) {
    if (!e || nclips <= 0 || !clip_len || !pose_host || !shape_host) return fail("uhc_load_clips_smpl: bad argument");
    if (pose_dim != 72 && pose_dim != 156) return fail("uhc_load_clips_smpl: pose_dim must be 72 (SMPL) or 156 (SMPL-H)");
    EngineKin kin;
    uhc_engine_kin(e, &kin);
    size_t total = 0;
    for (int c = 0; c < nclips; c++) {
        if (clip_len[c] < 2) return fail("uhc_load_clips_smpl: clip shorter than 2 frames");
        if (clip_model_host && (clip_model_host[c] < 0 || clip_model_host[c] >= kin.nshape)) return fail("uhc_load_clips_smpl: clip_model out of range");
        total += clip_len[c];
    }
    if (total * uhc_motion::REC > (size_t)1 << 40 || total > 0x7fffffff) return fail("uhc_load_clips_smpl: too many frames");
    for (size_t i = 0; i < (size_t)nclips * 17; i++) if (!isfinite(shape_host[i])) return fail("uhc_load_clips_smpl: non-finite shape value");
    CKM(cudaSetDevice(kin.device));
    return kin.precision == 32 ? build_table<float>(e, nclips, clip_len, pose_dim, pose_host, trans_host, shape_host, clip_model_host, kin, total)
                               : build_table<double>(e, nclips, clip_len, pose_dim, pose_host, trans_host, shape_host, clip_model_host, kin, total);
}

int uhc_get_clip_frames(UhcEngine *e, int frame0, int nframes, double *out_host) {
    if (!e || !out_host || frame0 < 0 || nframes <= 0) return fail("uhc_get_clip_frames: bad argument");
    EngineTable tb;
    if (uhc_engine_expert_table(e, &tb)) return -3;
    size_t total = 0;
    for (int c = 0; c < tb.num_clips; c++) total += tb.clip_len[c];
    if ((size_t)frame0 + nframes > total) return fail("uhc_get_clip_frames: rows outside the clip table");
    CKM(cudaSetDevice(tb.device));
    CKM(cudaDeviceSynchronize());
    const size_t n = (size_t)nframes * UHC_EX_SIZE, off = (size_t)frame0 * UHC_EX_SIZE;
    if (tb.precision == 64) { CKM(cudaMemcpy(out_host, (const double *)tb.expert + off, n * sizeof(double), cudaMemcpyDeviceToHost)); return 0; }
    std::vector<float> f(n);
    CKM(cudaMemcpy(f.data(), (const float *)tb.expert + off, n * sizeof(float), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; i++) out_host[i] = (double)f[i];
    return 0;
}

}  // extern "C"
