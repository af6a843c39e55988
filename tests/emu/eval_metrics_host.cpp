// host build of the metric stage (uhc_b200/csrc/eval_metrics.h) for the CPU test: the same per-row code the CUDA metric kernel runs
#include "../../uhc_b200/csrc/eval_metrics.h"

extern "C" void eval_metrics_host(const double *pq, const double *gq, const double *pj, const double *gj, int T, double *out) {
    for (int k = 0; k < T; k++) {
        const double *jp[3] = {pj + 72 * k, k >= 1 ? pj + 72 * (k - 1) : nullptr, k >= 2 ? pj + 72 * (k - 2) : nullptr};
        const double *jg[3] = {gj + 72 * k, k >= 1 ? gj + 72 * (k - 1) : nullptr, k >= 2 ? gj + 72 * (k - 2) : nullptr};
        uhc_eval::frame_metrics<double, double>(pq + 76 * k, gq + 76 * k, jp, jg, T, out + uhc_eval::NMET * k);
    }
}
