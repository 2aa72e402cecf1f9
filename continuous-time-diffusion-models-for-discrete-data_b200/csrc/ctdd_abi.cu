// C-ABI plumbing: error text, launch accounting, argument validation and kernel-family dispatch.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include "ctdd_common.cuh"

namespace ctdd {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int launch_step_simt(const ctdd_step_params* p, cudaStream_t st);
int launch_step_tc(const ctdd_step_params* p, cudaStream_t st);
int launch_step_tcq(const ctdd_step_params* p, cudaStream_t st);
bool tc_supports(const ctdd_step_params* p);
long long tc_workspace_bytes(long long rows, int S);

}  // namespace ctdd

extern "C" int ctdd_version(void) { return CTDD_ABI_VERSION; }
extern "C" const char* ctdd_last_error(void) { return ctdd::g_err; }
extern "C" long long ctdd_launch_count(void) { return ctdd::g_launches.load(); }

extern "C" int64_t ctdd_step_workspace_bytes(int64_t rows, int S, int impl) {
  if (impl == CTDD_IMPL_SIMT) return 0;
  return ctdd::tc_workspace_bytes(rows, S);
}

extern "C" int ctdd_reverse_step(const ctdd_step_params* p, void* stream) {
  using namespace ctdd;
  if (!p) { set_error("ctdd_reverse_step: null params"); return 2; }
  if (p->N <= 0 || p->D <= 0 || p->S < 2) { set_error("ctdd_reverse_step: bad sizes N=%d D=%d S=%d", p->N, p->D, p->S); return 2; }
  if (p->mode < CTDD_MODE_TAU_LEAP || p->mode > CTDD_MODE_EXACT) { set_error("ctdd_reverse_step: unknown mode %d", p->mode); return 2; }
  if (p->branch < CTDD_BRANCH_TAULDR || p->branch > CTDD_BRANCH_SDDM_REVERSE_LOGSCALE) { set_error("ctdd_reverse_step: unknown branch %d", p->branch); return 2; }
  if (p->head < CTDD_HEAD_LOGITS || p->head > CTDD_HEAD_LOGISTIC_FIX) { set_error("ctdd_reverse_step: unknown head %d", p->head); return 2; }
  if (p->head == CTDD_HEAD_LOGITS && p->logits_dtype != CTDD_DTYPE_F32 && p->logits_dtype != CTDD_DTYPE_BF16) {
    set_error("ctdd_reverse_step: unknown logits_dtype %d (CTDD_DTYPE_F32 = 0, CTDD_DTYPE_BF16 = 1)", p->logits_dtype);
    return 2;
  }
  if (p->head != CTDD_HEAD_LOGITS && p->head_dtype != CTDD_DTYPE_F32 && p->head_dtype != CTDD_DTYPE_BF16) {
    set_error("ctdd_reverse_step: unknown head_dtype %d (CTDD_DTYPE_F32 = 0, CTDD_DTYPE_BF16 = 1)", p->head_dtype);
    return 2;
  }
  if (p->head == CTDD_HEAD_LOGITS ? !p->logits : (!p->head_mu || !p->head_log_scale || p->head_batch_stride < p->D)) {
    set_error("ctdd_reverse_step: null logits (or head_mu / head_log_scale / head_batch_stride < D for a logistic head)");
    return 2;
  }
  if (!p->x_eval || !p->Rb || !p->RbT) { set_error("ctdd_reverse_step: null input pointer"); return 2; }
  if ((p->branch != CTDD_BRANCH_SDDM_DIRECT || p->mode == CTDD_MODE_EXACT) && (!p->Q || !p->QT)) { set_error("ctdd_reverse_step: Q/QT required for this branch"); return 2; }
  if (p->mode != CTDD_MODE_RATES_ONLY && !p->x_out) { set_error("ctdd_reverse_step: x_out is null"); return 2; }
  if (p->mode == CTDD_MODE_RATES_ONLY && !p->rr_out && !p->ratio_out) { set_error("ctdd_reverse_step: RATES_ONLY needs rr_out or ratio_out"); return 2; }
  if (p->head == CTDD_HEAD_LOGITS && p->ld_logits < p->S) { set_error("ctdd_reverse_step: ld_logits < S"); return 2; }
  if (p->row_offset & 7) { set_error("ctdd_reverse_step: row_offset must be a multiple of 8 (got %lld)", (long long)p->row_offset); return 2; }
  if ((p->tc_tables != nullptr) != (p->tc_static != nullptr)) {
    set_error("ctdd_reverse_step: tc_tables and tc_static must be given together (got only one); refusing to fall back silently");
    return 2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool want_tc = (p->impl == CTDD_IMPL_TC) || (p->impl == CTDD_IMPL_AUTO && tc_supports(p));
  if (want_tc) {
    if (!tc_supports(p)) { set_error("ctdd_reverse_step: tcgen05 path does not support S=%d mode=%d branch=%d (or tc_tables/workspace missing)", p->S, p->mode, p->branch); return 3; }
    // Euler modes need a row's total rate before its one pick: the row-gather kernel; every other mode: chunk-local
    if (p->mode == CTDD_MODE_EULER || p->mode == CTDD_MODE_EULER_CORR) return launch_step_tc(p, st);
    return launch_step_tcq(p, st);
  }
  if (p->head != CTDD_HEAD_LOGITS) {
    set_error("ctdd_reverse_step: the fused logistic head exists on the tcgen05 path only (S == 256, tc tables given); "
              "materialise the logits with ctdd_logistic_logits for S=%d mode=%d branch=%d", p->S, p->mode, p->branch);
    return 3;
  }
  return launch_step_simt(p, st);
}
