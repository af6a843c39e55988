// eval.cu -- policy evaluation behind the C ABI (include/uhc_eval.h): uhc_evaluate, uhc_eval_metrics.
//
// Replaces the host loop of AgentCopycat.eval_policy (uhc/agents/agent_copycat.py:354-494: per control step policy -> env.step -> three
// blocking reads of fail / end / reward, a state gather, fail_safe through set_state, then numpy metrics per clip) by
//   a work queue of clips over the E env slots: a slot whose episode ends takes the next clip inside the step kernel (k_env_step<.., true>,
//     env_step.h eval_after_step), an idle slot runs no physics;
//   K = 16 control steps per CUDA graph replay (ZFilter without update -> policy GEMMs -> mean action: uhc_policy_forward's kernels, then the
//     eval-mode step kernel); the host reads the number of active slots between replays;
//   one fp64 metric kernel over every recorded row (eval_metrics.h), one CTA per clip, the per-clip means reduced in the same CTA.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/uhc_b200.h"
#include "../../include/uhc_rollout.h"
#include "../../include/uhc_eval.h"
#include "sim_core.h"
#include "env_step.h"
#include "eval_internal.h"
#include "eval_metrics.h"

static thread_local std::string g_ev_err;
#define CKE(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { g_ev_err = std::string(#x) + ": " + cudaGetErrorString(e_); return -1; } } while (0)

namespace {

constexpr int STEPS_PER_GRAPH = 16;
constexpr int MET_THREADS = 128;

// ---- metric stage: one CTA per clip; thread k scores rows k, k + 128, ...; then the per-clip means (fixed reduction order)
struct GtRows {      // ground truth of a row: explicit arrays (uhc_eval_metrics) or the engine's expert table at min(frame_t, len - 1)
    const void *q, *j;                                   // explicit: [F][76], [F][72] double
    const void *expert; const int *clip_adr; int clip0; const int *frame_t;   // expert table (float or double)
};
template <class P, class G, bool TABLE>
__global__ void __launch_bounds__(MET_THREADS)
k_eval_metrics(const P *__restrict__ pq, const P *__restrict__ pj, GtRows gt, const int *__restrict__ frame_off, const int *__restrict__ nframes,
               int n, double *__restrict__ fm, double *__restrict__ cm) {
    using namespace uhc_eval;
    const int i = blockIdx.x;
    if (i >= n) return;
    const int r0 = frame_off[i], T = nframes ? nframes[i] : frame_off[i + 1] - frame_off[i];
    int base = 0, len = 0;
    if (TABLE) { base = gt.clip_adr[gt.clip0 + i]; len = gt.clip_adr[gt.clip0 + i + 1] - base; }
    auto grow = [&](int k, const G **q, const G **j) {
        if (TABLE) {
            const int t = gt.frame_t[r0 + k];
            const G *f = (const G *)gt.expert + (size_t)(base + (t < len - 1 ? t : len - 1)) * uhc::EX_SIZE;
            *q = f + uhc::EX_QPOS; *j = f + uhc::EX_WBPOS;
        } else { *q = (const G *)gt.q + (size_t)(r0 + k) * 76; *j = (const G *)gt.j + (size_t)(r0 + k) * 72; }
    };
    double acc[NMET] = {0, 0, 0, 0, 0, 0};
    for (int k = threadIdx.x; k < T; k += blockDim.x) {
        const P *jp[3] = {pj + (size_t)(r0 + k) * 72, k >= 1 ? pj + (size_t)(r0 + k - 1) * 72 : nullptr, k >= 2 ? pj + (size_t)(r0 + k - 2) * 72 : nullptr};
        const G *qg, *jg[3] = {nullptr, nullptr, nullptr};
        grow(k, &qg, &jg[0]);
        for (int d = 1; d <= 2 && d <= k; d++) { const G *qd; grow(k - d, &qd, &jg[d]); }
        double m[NMET];
        frame_metrics<P, G>(pq + (size_t)(r0 + k) * 76, qg, jp, jg, T, m);
        for (int c = 0; c < NMET; c++) {
            fm[(size_t)(r0 + k) * NMET + c] = m[c];
            if (!(c == M_VEL && k < 1) && !(c == M_ACCEL && k < 2)) acc[c] += m[c];
        }
    }
    __shared__ double red[NMET][MET_THREADS];
    for (int c = 0; c < NMET; c++) red[c][threadIdx.x] = acc[c];
    __syncthreads();
    for (int s = MET_THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) for (int c = 0; c < NMET; c++) red[c][threadIdx.x] += red[c][threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x < NMET) {
        const int c = threadIdx.x, cnt = T - (c == M_VEL ? 1 : (c == M_ACCEL ? 2 : 0));
        cm[(size_t)i * NMET + c] = T < 3 ? (double)NAN : red[c][0] / (double)cnt;
    }
}

// slot s < m starts on clip s of the range, the others idle; per-clip outputs zeroed
__global__ void k_eval_init(int *slot_clip, int *slot_k, int *queue, int E, int m, int n, int *nframes, int *last_t, int *fail_any, double *reward_sum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < E) { slot_clip[i] = i < m ? i : -1; slot_k[i] = 0; }
    if (i < n) { nframes[i] = 0; last_t[i] = 0; fail_any[i] = 0; reward_sum[i] = 0.0; }
    if (i == 0) { queue[0] = m; queue[1] = m; queue[2] = 0; }
}
// queue[2] counts the control steps that start with an active slot (the replays of the last graph run idle steps past the end)
__global__ void k_eval_count(int *queue) { if (queue[1] > 0) queue[2] += 1; }

// per-engine scratch of the loop (owned here, not by the engine).  The step graph is NOT kept between calls: it holds the engine's view
// (clip table, configuration) and the policy scratch of rollout.cu by value, and any uhc_load_clips / uhc_engine_set_cfg / rollout between
// two calls may replace them; capturing 16 steps costs far less than one evaluation.
struct EvalCtx {
    UhcEngine *eng = nullptr; int E = 0, D = 0, A = 0, device = -1;
    float *obs = nullptr, *act = nullptr, *rew = nullptr; int *fail = nullptr, *end = nullptr; unsigned char *det = nullptr;
    int *slot_clip = nullptr, *slot_k = nullptr, *queue = nullptr; int *h_active = nullptr;
    long long last_steps = 0;
};
std::vector<EvalCtx *> g_ectx;

void free_ctx(EvalCtx *c) {
    for (void *p : {(void *)c->obs, (void *)c->act, (void *)c->rew, (void *)c->fail, (void *)c->end, (void *)c->det, (void *)c->slot_clip, (void *)c->slot_k, (void *)c->queue})
        if (p) cudaFree(p);
    if (c->h_active) cudaFreeHost(c->h_active);
    c->obs = c->act = c->rew = nullptr; c->fail = c->end = c->slot_clip = c->slot_k = c->queue = c->h_active = nullptr; c->det = nullptr;
}

int ctx_of(UhcEngine *e, int device, EvalCtx **out) {
    EvalCtx *c = nullptr;
    for (EvalCtx *x : g_ectx) if (x->eng == e) c = x;
    if (!c) { c = new EvalCtx(); c->eng = e; g_ectx.push_back(c); }
    const int E = uhc_num_envs(e), D = uhc_engine_obs_dim(e), A = uhc_engine_act_dim(e);
    if (c->E != E || c->D != D || c->A != A || c->device != device) {       // (re)size the scratch: obs / action / step outputs of every slot, the queue
        free_ctx(c);
        c->E = E; c->D = D; c->A = A; c->device = device;
        CKE(cudaMalloc((void **)&c->obs, (size_t)E * D * 4)); CKE(cudaMalloc((void **)&c->act, (size_t)E * A * 4)); CKE(cudaMalloc((void **)&c->rew, (size_t)E * 4));
        CKE(cudaMalloc((void **)&c->fail, (size_t)E * 4)); CKE(cudaMalloc((void **)&c->end, (size_t)E * 4)); CKE(cudaMalloc((void **)&c->det, (size_t)E));
        CKE(cudaMalloc((void **)&c->slot_clip, (size_t)E * 4)); CKE(cudaMalloc((void **)&c->slot_k, (size_t)E * 4)); CKE(cudaMalloc((void **)&c->queue, 3 * 4));
        CKE(cudaHostAlloc((void **)&c->h_active, 2 * 4, cudaHostAllocDefault));
        CKE(cudaMemset(c->det, 1, (size_t)E));      // every action is the policy mean
        CKE(cudaMemset(c->obs, 0, (size_t)E * D * 4));
    }
    *out = c;
    return 0;
}

int policy_step(EvalCtx *c, const UhcMlp *mlp, const UhcMcp *mcp, const float *log_std, const double *zstats, float zclip, cudaStream_t st) {
    const int rc = mcp ? uhc_policy_forward_mcp(c->eng, c->obs, mcp, log_std, (double *)zstats, zclip, 0, 0ull, c->det, nullptr, c->act, nullptr, st)
                       : uhc_policy_forward(c->eng, c->obs, mlp, log_std, (double *)zstats, zclip, 0, 0ull, c->det, nullptr, c->act, nullptr, st);
    if (rc) { g_ev_err = std::string("policy: ") + uhc_rollout_last_error(); return rc; }
    return 0;
}

int launch_metrics(const EngineTable &tab, int clip0, int n, const UhcEvalBuf *b, cudaStream_t st) {
    GtRows gt; memset(&gt, 0, sizeof gt);
    gt.expert = tab.expert; gt.clip_adr = tab.clip_adr; gt.clip0 = clip0; gt.frame_t = b->frame_t;
    if (tab.precision == 32) k_eval_metrics<float, float, true><<<n, MET_THREADS, 0, st>>>(b->pred_qpos, b->pred_jpos, gt, b->frame_off, b->nframes, n, b->frame_metrics, b->clip_metrics);
    else k_eval_metrics<float, double, true><<<n, MET_THREADS, 0, st>>>(b->pred_qpos, b->pred_jpos, gt, b->frame_off, b->nframes, n, b->frame_metrics, b->clip_metrics);
    CKE(cudaGetLastError());
    return 0;
}

int evaluate_impl(UhcEngine *e, int clip0, int n, const UhcMlp *mlp, const UhcMcp *mcp, const float *log_std, const double *zstats, float zclip,
                  int fail_safe, const UhcEvalBuf *b, void *stream, const char *who) {
    const std::string w(who);
    if (!e || (!mlp && !mcp) || !log_std || !zstats || !b) { g_ev_err = w + ": bad argument"; return -2; }
    if (!b->frame_off || !b->pred_qpos || !b->pred_jpos || !b->frame_t || !b->frame_metrics || !b->nframes || !b->last_t || !b->fail_any ||
        !b->reward_sum || !b->clip_metrics) { g_ev_err = w + ": missing buffer in UhcEvalBuf"; return -2; }
    EngineTable tab;
    if (uhc_engine_expert_table(e, &tab)) { g_ev_err = w + ": no clips loaded"; return -3; }
    if (n <= 0 || clip0 < 0 || clip0 + n > tab.num_clips) {
        g_ev_err = w + ": clip range [" + std::to_string(clip0) + ", " + std::to_string(clip0 + n) + ") is not inside the loaded table of " + std::to_string(tab.num_clips) + " clips";
        return -2;
    }
    CKE(cudaSetDevice(tab.device));
    cudaStream_t st = (cudaStream_t)stream;
    // the offset table must give every clip its len - 1 + trail_steps rows inside frame_cap
    std::vector<int> off(n + 1);
    CKE(cudaMemcpyAsync(off.data(), b->frame_off, (n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CKE(cudaStreamSynchronize(st));
    long long rows = 0;
    for (int i = 0; i < n; i++) {
        const int need = tab.clip_len[clip0 + i] - 1 + (tab.trail_steps > 0 ? tab.trail_steps : 0);
        if (off[0] < 0 || off[i + 1] - off[i] < need) {
            g_ev_err = w + ": frame_off gives clip " + std::to_string(i) + " " + std::to_string(off[i + 1] - off[i]) + " rows, it needs len - 1 + trail_steps = " + std::to_string(need);
            return -2;
        }
        rows += need;
    }
    if (off[n] > b->frame_cap) { g_ev_err = w + ": frame_off[n] = " + std::to_string(off[n]) + " exceeds frame_cap = " + std::to_string(b->frame_cap); return -2; }
    EvalCtx *c;
    if (ctx_of(e, tab.device, &c)) return -1;
    const int E = c->E, m = n < E ? n : E;
    uhc::EvalView xv; memset(&xv, 0, sizeof xv);
    xv.clip0 = clip0; xv.n = n; xv.fail_safe = fail_safe ? 1 : 0; xv.frame_off = b->frame_off; xv.pred_qpos = b->pred_qpos; xv.pred_jpos = b->pred_jpos;
    xv.frame_t = b->frame_t; xv.nframes = b->nframes; xv.last_t = b->last_t; xv.fail_any = b->fail_any; xv.reward_sum = b->reward_sum;
    xv.slot_clip = c->slot_clip; xv.slot_k = c->slot_k; xv.queue = c->queue;
    const int g = (E > n ? E : n);
    k_eval_init<<<(g + 255) / 256, 256, 0, st>>>(c->slot_clip, c->slot_k, c->queue, E, m, n, b->nframes, b->last_t, b->fail_any, b->reward_sum);
    CKE(cudaGetLastError());
    {   // slot s <- clip clip0 + s, frame 0: the reset kernel of uhc_env_reset with auto_reset cleared (no reactive standing-neutral starts),
        // the same reset the queue runs in the step kernel for the later clips
        std::vector<int> ids(m), clip(m), start(m, 0), len(m);
        for (int s = 0; s < m; s++) { ids[s] = s; clip[s] = clip0 + s; len[s] = tab.clip_len[clip0 + s]; }
        if (uhc_env_reset_eval(e, m, ids.data(), clip.data(), start.data(), len.data(), c->obs, st)) { g_ev_err = w + ": reset: " + uhc_last_error(); return -1; }
    }
    if (policy_step(c, mlp, mcp, log_std, zstats, zclip, st)) return -1;     // sizes the policy scratch outside the capture
    cudaGraphExec_t exec = nullptr;
    {
        cudaStream_t cs; CKE(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        CKE(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        int rc = 0;
        for (int k = 0; k < STEPS_PER_GRAPH && !rc; k++) {
            k_eval_count<<<1, 1, 0, cs>>>(c->queue);
            rc = policy_step(c, mlp, mcp, log_std, zstats, zclip, cs);
            if (!rc && uhc_env_step_eval(e, c->act, c->obs, c->rew, c->fail, c->end, xv, cs)) { g_ev_err = w + ": env step: " + uhc_last_error(); rc = -1; }
        }
        cudaError_t ce = cudaStreamEndCapture(cs, &graph);
        cudaStreamDestroy(cs);
        if (rc) { if (graph) cudaGraphDestroy(graph); return -1; }
        if (ce != cudaSuccess) { g_ev_err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce); return -1; }
        ce = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { g_ev_err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce); return -1; }
    }
    // every step of an active slot records a row: the loop cannot need more steps than rows
    long long replays = 0;
    cudaError_t ce = cudaSuccess;
    for (;;) {
        if ((ce = cudaGraphLaunch(exec, st)) != cudaSuccess) break;
        if ((ce = cudaMemcpyAsync(c->h_active, c->queue + 1, 2 * sizeof(int), cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        if ((ce = cudaStreamSynchronize(st)) != cudaSuccess) break;
        replays++;
        if (c->h_active[0] == 0) break;
        if (replays * STEPS_PER_GRAPH > rows + STEPS_PER_GRAPH) break;
    }
    cudaGraphExecDestroy(exec);
    if (ce != cudaSuccess) { g_ev_err = w + ": step graph: " + cudaGetErrorString(ce); return -1; }
    if (c->h_active[0] != 0) { g_ev_err = w + ": slots still active after " + std::to_string(replays * STEPS_PER_GRAPH) + " steps for " + std::to_string(rows) + " rows"; return -1; }
    const long long steps = c->h_active[1];
    c->last_steps = steps;
    return launch_metrics(tab, clip0, n, b, st);
}

}  // namespace

extern "C" {

const char *uhc_eval_last_error(void) { return g_ev_err.c_str(); }

int uhc_evaluate(UhcEngine *e, int clip0, int n, const UhcMlp *mlp, const float *log_std, const double *zfilter_stats, float zclip,
                 int fail_safe, const UhcEvalBuf *out, void *stream) {
    if (!mlp) { g_ev_err = "uhc_evaluate: bad argument"; return -2; }
    return evaluate_impl(e, clip0, n, mlp, nullptr, log_std, zfilter_stats, zclip, fail_safe, out, stream, "uhc_evaluate");
}
int uhc_evaluate_mcp(UhcEngine *e, int clip0, int n, const UhcMcp *mcp, const float *log_std, const double *zfilter_stats, float zclip,
                     int fail_safe, const UhcEvalBuf *out, void *stream) {
    if (!mcp) { g_ev_err = "uhc_evaluate_mcp: bad argument"; return -2; }
    return evaluate_impl(e, clip0, n, nullptr, mcp, log_std, zfilter_stats, zclip, fail_safe, out, stream, "uhc_evaluate_mcp");
}

int uhc_eval_last_steps(UhcEngine *e, long long *steps_host) {
    if (!e || !steps_host) { g_ev_err = "uhc_eval_last_steps: bad argument"; return -2; }
    *steps_host = 0;
    for (EvalCtx *c : g_ectx) if (c->eng == e) *steps_host = c->last_steps;
    return 0;
}

int uhc_eval_metrics(const double *pred_qpos, const double *gt_qpos, const double *pred_jpos, const double *gt_jpos, const int *frame_off,
                     const int *nframes, int n, double *frame_metrics, double *clip_metrics, void *stream) {
    if (!pred_qpos || !gt_qpos || !pred_jpos || !gt_jpos || !frame_off || !frame_metrics || !clip_metrics) { g_ev_err = "uhc_eval_metrics: missing buffer"; return -2; }
    if (n <= 0) { g_ev_err = "uhc_eval_metrics: n <= 0"; return -2; }
    GtRows gt; memset(&gt, 0, sizeof gt);
    gt.q = gt_qpos; gt.j = gt_jpos;
    k_eval_metrics<double, double, false><<<n, MET_THREADS, 0, (cudaStream_t)stream>>>(pred_qpos, pred_jpos, gt, frame_off, nframes, n, frame_metrics, clip_metrics);
    CKE(cudaGetLastError());
    return 0;
}

void uhc_eval_release(UhcEngine *e) {
    for (size_t i = 0; i < g_ectx.size(); i++) if (g_ectx[i]->eng == e) {
        free_ctx(g_ectx[i]); delete g_ectx[i]; g_ectx.erase(g_ectx.begin() + i); return;
    }
}

}  // extern "C"
