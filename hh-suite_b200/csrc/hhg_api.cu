// hh-suite_b200/csrc/hhg_api.cu -- the C-ABI (include/hhg.h) over the sm_100a kernels.
// Host side: planning (length-sorted 32-target warp jobs, strip work items, memory waves),
// device memory, launches.  There is no CPU fallback: without a CUDA device every entry point fails.
#include "../../include/hhg.h"
#include "hhg_kernels.cuh"
#include "hhg_hhm.cuh"
#include "hhg_msa.cuh"
#include "hhg_crf.cuh"
#include "hhg_mac.cuh"
#include "hhg_topk.cuh"
#include "hhg_hitlist.h"

#include <dlfcn.h>
#if defined(__SSE__)
#include <xmmintrin.h>     // RCPPS: the alignment weights of the reference go through it (hhg_msa.cuh)
#endif

#include <algorithm>
#include <chrono>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <cmath>
#include <cfloat>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

using namespace hhg;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(expr)                                                                                  \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess)                                                                       \
      return fail(e__ == cudaErrorMemoryAllocation ? HHG_ENOMEM : HHG_ECUDA, "%s: %s (%s:%d)", #expr, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                   \
  } while (0)

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  cudaError_t alloc(size_t count) {
    release();
    n = count;
    if (count == 0) return cudaSuccess;
    return cudaMalloc((void**)&p, count * sizeof(T));
  }
  cudaError_t ensure(size_t count) {
    if (count <= n && p) return cudaSuccess;
    return alloc(count);
  }
};

// strip height forced by the environment (developer / test knob), or 0 = chosen per plan (plan_strip_rows)
int strip_rows() {
  const char* e = getenv("HHG_STRIP_ROWS");
  if (e) {
    int r = atoi(e);
    if (r == 8 || r == 12 || r == 16) return r;
  }
  return 0;
}

}  // namespace

struct hhg_ctx {
  int device = 0;
  std::shared_ptr<void> msa_cache;     // MsaChunk reused by the single-alignment calls (hhg_msa_to_hmm, hhg_query_from_a3m)
  std::shared_ptr<void> crf_cache;     // device + pinned host staging of hhg_query_context_pseudocounts
  std::shared_ptr<void> msa_rcp;       // DevBuf<float>: the host's RCPPS table (hhg_msa.cuh), uploaded once per context
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 0;
  long long launches = 0;
  // query
  int Lq = 0, R = 0;     // Lq: length of query 0; R: forced strip height (HHG_STRIP_ROWS) or 0 = per plan
  // query batch (hhg_query_set = a batch of one): lengths, first row record of each query in qrec, average aa
  // frequencies (for the fused null model of batch searches over a raw shard)
  int nq = 0;
  std::vector<int> q_L, q_row0;
  std::vector<float> h_q_pav;
  bool has_q_pav = false;
  DevBuf<float> d_q_pav, d_pb;
  // excluded regions (-excl / -template_excl), applied to every search until cleared
  std::vector<int> ex_q_lo, ex_q_hi, ex_t_lo, ex_t_hi;
  DevBuf<int> d_ex;
  unsigned long long query_serial = 0;   // bumped by every hhg_query_set*: plans built for an older batch are rebuilt
  int group_jobs = 16;   // work-item interleave (see k_viterbi): 16 jobs x nstrips items keep the group L2-resident
  uint32_t epoch = 0;    // run counter feeding the boundary-slot tags
  uint32_t epoch_window = 1;   // number of times the 20-bit epoch has wrapped (+1)
  DevBuf<float4> qrec;
  DevBuf<float> S33;
  DevBuf<float> lg2, diff;   // fast_log2 tables for Hit.score
  std::vector<float> h_lg2;
  bool has_ss = false, has_S33 = false;
  hhg_params par{1, 0.f, 0.f, -0.03f, 0.11f, 0, 0.1f, 2};
  // prefilter
  DevBuf<uint8_t> pf_prof, sw_prof;
  DevBuf<uint8_t> pf_edge[2];   // per-column hand-off between query tiles of the ungapped prefilter (Lq > 512)
  DevBuf<int> sw_ids, sw_scores;
  DevBuf<unsigned> pf_counter, pf_hist;
  DevBuf<int> pf_corr, pf_ids_a, pf_score_a, pf_ids_b;
  // MAC realignment (hhg_mac_*): query in linear transition space + grow-only scratch of the last call
  int mac_Lq = 0;
  DevBuf<float> mac_qp, mac_qtr, mac_ttr, mac_post, mac_out_post;
  DevBuf<uint8_t> mac_off, mac_bt, mac_out_states;
  DevBuf<double> mac_rows, mac_scale;
  DevBuf<long long> mac_i64, mac_dbg;
  DevBuf<int> mac_i32, mac_out_i, mac_out_j, mac_map;
  cudaStream_t aux_stream = nullptr;     // long-template launch of hhg_mac_realign
  cudaEvent_t aux_ev[2] = {nullptr, nullptr};
  DevBuf<MacHitOut> mac_out;
  std::vector<long long> mac_cell_off;   // of the last call (debug fetch)
  std::vector<int> mac_Lt;
  size_t max_bt_bytes = 0;   // memory-wave budget for backtrace words
  struct hhg_plan* scratch_plan = nullptr;   // reused by hhg_viterbi_search
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

static std::atomic<unsigned long long> g_db_serial{1};

struct hhg_db {
  const unsigned long long serial = g_db_serial.fetch_add(1);   // identity for plan reuse (addresses get recycled)
  int device = 0;
  int n = 0;
  long long total_cols = 0;
  bool has_ss = false;
  std::vector<int> L;
  std::vector<long long> col_off;
  DevBuf<int> dL;
  DevBuf<long long> dcol_off;
  DevBuf<float4> cols;       // prepared column records (what the DP reads)
  bool raw = false;          // created by hhg_db_create_raw: cols is filled by hhg_db_apply_null_model
  DevBuf<float4> cols_raw;   // pre-null-model records
  DevBuf<float> pav;         // [n*20] template average aa frequencies
  bool prepared = true;
  unsigned long long cols_version = 1;   // bumped whenever `cols` is rewritten (hhg_db_apply_null_model)
};

struct hhg_csdb {
  int device = 0;
  int n = 0;
  long long total = 0;
  DevBuf<int> dL;
  DevBuf<long long> doff;
  DevBuf<uint8_t> seq;
  DevBuf<int> scores;
};

struct Wave {
  int job_begin = 0, job_end = 0;
  long long item_begin = 0, item_end = 0;   // slice of the plan's work-item table (job index relative to job_begin)
};

struct hhg_plan {
  const hhg_db* db = nullptr;
  unsigned long long db_serial = 0;
  int device = 0;
  int n = 0;            // requests
  int Lq = 0, R = 16;   // Lq: length of query 0 (single-query callers)
  std::vector<int> q_L, q_row0;          // query batch geometry the plan was built for
  std::vector<int> req_query;            // request -> query index
  int njobs = 0;
  long long ss_total = 0, co_total = 0;  // per-strip maxima blocks / cell-off words over all jobs
  double cells = 0, padded_cells = 0, alg_bytes = 0;
  std::vector<int> ids;          // request -> target id
  std::vector<int> order;        // sorted position -> request index
  std::vector<int> req_job, req_lane;   // per request
  std::vector<int> job_Lmax, job_query, job_nstrips, job_Lq, job_qrow0;
  std::vector<long long> job_ss_off;
  std::vector<int2> items;
  std::vector<long long> job_bt_off, job_bnd_off, job_co_off, job_jc_off, path_off;
  long long jc_total = 0;                 // float4 in the job-interleaved operand stream
  unsigned long long jc_version = 0;      // db->cols_version the stream was built from (0 = never)
  int nm_mode = -1;                       // >= 0: columnscore of the null model fused into the stream (raw shard)
  int jc_nm_mode = -2;                    // nm_mode / query batch the stream was built with
  unsigned long long jc_query_serial = 0;
  std::vector<Wave> waves;
  long long path_total = 0;
  // device
  DevBuf<int> d_job_target, d_job_Lmax, d_req_job, d_req_lane, d_req_Lt, d_req_Lq, d_req_target;
  DevBuf<int> d_job_query, d_job_nstrips, d_job_Lq, d_job_qrow0;
  DevBuf<long long> d_job_ss_off;
  DevBuf<int2> d_items;
  DevBuf<float> d_S;
  DevBuf<long long> d_job_bt_off, d_job_bnd_off, d_job_co_off, d_job_jc_off, d_path_off;
  DevBuf<float4> d_jcols;
  DevBuf<uint32_t> d_bt, d_co;
  DevBuf<BndSlot> d_bnd;
  uint32_t bnd_epoch_window = 0;   // epoch window in which d_bnd was last cleared
  DevBuf<float> d_strip_score;
  DevBuf<int> d_strip_ij;
  DevBuf<unsigned> d_counter;
  float ms_viterbi = 0, ms_backtrace = 0;   // filled by hhg_plan_run_timed
  size_t max_bt_bytes = 0;
  DevBuf<uint8_t> d_paths_compact;
  DevBuf<long long> d_compact_off;
  std::vector<long long> h_compact_off;
  DevBuf<HitRec> d_hits;
  // top-K selection / exchange scratch (hhg_plan_topk)
  DevBuf<unsigned long long> d_keys;
  DevBuf<int> d_gids;
  DevBuf<float> d_user_key;
  DevBuf<TopkState> d_topk_state;
  DevBuf<TopkRec> d_topk_local, d_topk_all;
  DevBuf<uint8_t> d_topk_paths;
  DevBuf<uint8_t> d_paths;
  // cell-off input (optional)
  bool celloff = false;
  int n_excl_steps = 0;
  DevBuf<int> d_step_req, d_step_i, d_step_j;
};

extern "C" {

int hhg_plan_destroy(hhg_plan* plan);

const char* hhg_last_error(void) { return g_err.c_str(); }

int hhg_ctx_create(int device, void* stream, hhg_ctx** out) {
  if (!out) return fail(HHG_EINVAL, "out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(HHG_ENODEV, "no CUDA device available (%s); this library has no CPU fallback",
                cudaGetErrorString(e));
  if (device < 0) CK(cudaGetDevice(&device));
  if (device >= ndev) return fail(HHG_EINVAL, "device %d out of range (%d devices)", device, ndev);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  // sm_100a code only loads on compute capability 10.0; the fence-free 256-bit slot hand-off of k_viterbi was
  // validated on exactly that part (tests/test_kernel_variants_gpu.py stress test)
  if (prop.major != 10 || prop.minor != 0)
    return fail(HHG_ENODEV, "device %d is sm_%d%d; this library is built and validated for sm_100a (B200) only", device,
                prop.major, prop.minor);
  std::unique_ptr<hhg_ctx> holder(new hhg_ctx());
  hhg_ctx* c = holder.get();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (stream) {
    c->stream = (cudaStream_t)stream;
  } else {
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  c->R = strip_rows();
  {
    // fast_log2 tables exactly as the reference fills them on first use (src/util-inl.h:113-121):
    // lg2[i] = log2(1 + i/1024) via the C library's double-precision log (that is the overload the
    // reference's expression resolves to; verified against its table), diff[i] = slope / 8096
    std::vector<float> lg2(1025, 0.f), diff(1025, 0.f);
    float prev = 0.0f;
    for (int i = 1; i <= 1024; ++i) {
      lg2[i] = (float)(::log((double)(1024 + i)) * 1.442695041 - 10.0);
      diff[i - 1] = (float)((double)(lg2[i] - prev) * 1.2352E-4);
      prev = lg2[i];
    }
    c->h_lg2 = lg2;
    cudaError_t e1 = c->lg2.alloc(1025), e2 = c->diff.alloc(1025);
    if (e1 != cudaSuccess || e2 != cudaSuccess) return fail(HHG_ENOMEM, "fast_log2 tables");
    CK(cudaMemcpy(c->lg2.p, lg2.data(), 1025 * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->diff.p, diff.data(), 1025 * 4, cudaMemcpyHostToDevice));
  }
  { const char* ge = getenv("HHG_GROUP_JOBS"); c->group_jobs = ge ? std::max(1, atoi(ge)) : 16; }
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  const char* env = getenv("HHG_MAX_BT_GB");
  double cap = env ? atof(env) * 1e9 : 48e9;
  c->max_bt_bytes = (size_t)std::min(cap, 0.45 * (double)free_b);
  *out = holder.release();
  return HHG_OK;
}

int hhg_ctx_destroy(hhg_ctx* ctx) {
  if (!ctx) return HHG_OK;
  cudaSetDevice(ctx->device);
  if (ctx->scratch_plan) hhg_plan_destroy(ctx->scratch_plan);
  for (auto& e : ctx->ev) if (e) cudaEventDestroy(e);
  for (auto& e : ctx->aux_ev) if (e) cudaEventDestroy(e);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return HHG_OK;
}

int hhg_ctx_sync(hhg_ctx* ctx) {
  if (!ctx) return fail(HHG_EINVAL, "ctx is NULL");
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

long long hhg_ctx_launch_count(hhg_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------ DB
static int pack_profiles(hhg_ctx* ctx, int n, const int32_t* L, const int64_t* p_off,
                         const int64_t* tr_off, const int64_t* ss_off, const float* p, const float* tr,
                         const uint8_t* ss, const std::vector<long long>& col_off, long long total_cols,
                         float4* d_out) {
  // upload the raw profiles in bounded chunks of targets, pack on the device
  const size_t kChunkBytes = (size_t)1 << 30;
  DevBuf<float> dp, dtr;
  DevBuf<uint8_t> dss;
  DevBuf<int> dL;
  DevBuf<long long> dcol, dpo, dto, dso;
  int t0 = 0;
  while (t0 < n) {
    // the profiles of consecutive targets need not be contiguous in the caller's arrays; upload per
    // target range [lo, hi) covering min..max offsets when contiguous, else target by target.
    int t1 = t0;
    size_t bytes = 0;
    while (t1 < n && (bytes == 0 || bytes + (size_t)(L[t1] + 2) * 80 < kChunkBytes)) {
      bytes += (size_t)(L[t1] + 2) * 80;
      ++t1;
    }
    const int m = t1 - t0;
    std::vector<long long> po(m), to(m), so(m), co(m);
    std::vector<int> LL(m);
    size_t np = 0, ntr = 0, nss = 0;
    for (int k = 0; k < m; ++k) {
      LL[k] = L[t0 + k];
      po[k] = (long long)np; to[k] = (long long)ntr; so[k] = (long long)nss;
      co[k] = col_off[t0 + k] - col_off[t0];
      np += (size_t)(LL[k] + 2) * 20; ntr += (size_t)(LL[k] + 1) * 7; nss += (size_t)(LL[k] + 2);
    }
    std::vector<float> hp(np), htr(ntr);
    std::vector<uint8_t> hss(ss ? nss : 0);
    for (int k = 0; k < m; ++k) {
      memcpy(hp.data() + po[k], p + p_off[t0 + k], (size_t)(LL[k] + 2) * 20 * sizeof(float));
      memcpy(htr.data() + to[k], tr + tr_off[t0 + k], (size_t)(LL[k] + 1) * 7 * sizeof(float));
      if (ss) memcpy(hss.data() + so[k], ss + ss_off[t0 + k], (size_t)(LL[k] + 2));
    }
    // emissions are probabilities (ratios): the forward kernel's dot product relies on them being >= 0 (-0.0 is fine)
    for (int k = 0; k < m; ++k) {
      const float* row = hp.data() + po[k] + 20;
      for (int a = 0; a < LL[k] * 20; ++a)
        if (row[a] < 0.0f)
          return fail(HHG_EINVAL, "profile %d: emission %g at column %d is negative", t0 + k, row[a], a / 20 + 1);
    }
    const long long cols = (t1 < n ? col_off[t1] : total_cols) - col_off[t0];
    CK(dp.ensure(np)); CK(dtr.ensure(ntr)); CK(dL.ensure(m)); CK(dcol.ensure(m)); CK(dpo.ensure(m));
    CK(dto.ensure(m)); CK(dso.ensure(m));
    if (ss) CK(dss.ensure(nss));
    CK(cudaMemcpyAsync(dp.p, hp.data(), np * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dtr.p, htr.data(), ntr * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (ss) CK(cudaMemcpyAsync(dss.p, hss.data(), nss, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dL.p, LL.data(), m * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dcol.p, co.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dpo.p, po.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dto.p, to.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dso.p, so.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 128;
    const long long blocks = (cols + threads - 1) / threads;
    k_pack_cols<<<(unsigned)blocks, threads, 0, ctx->stream>>>(
        m, dL.p, dcol.p, dpo.p, dto.p, dso.p, dp.p, dtr.p, ss ? dss.p : nullptr,
        reinterpret_cast<ColRec*>(d_out) + col_off[t0], cols);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));   // host staging vectors die at scope end
    t0 = t1;
  }
  return HHG_OK;
}

int hhg_db_create(hhg_ctx* ctx, int n, const int32_t* L, const int64_t* p_off, const int64_t* tr_off,
                  const int64_t* ss_off, const float* p, const float* tr, const uint8_t* ss,
                  hhg_db** out) {
  if (!ctx || !out || n <= 0 || !L || !p_off || !tr_off || !p || !tr)
    return fail(HHG_EINVAL, "hhg_db_create: bad argument");
  if (ss && !ss_off) return fail(HHG_EINVAL, "hhg_db_create: ss given without ss_off");
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<hhg_db> holder(new hhg_db());   // freed on every early return below
  hhg_db* db = holder.get();
  db->device = ctx->device;
  db->n = n;
  db->has_ss = ss != nullptr;
  db->L.assign(L, L + n);
  db->col_off.resize(n);
  long long tot = 0;
  for (int k = 0; k < n; ++k) {
    if (L[k] < 1 || L[k] > 32767) return fail(HHG_EINVAL, "target %d: length %d out of [1,32767]", k, L[k]);
    db->col_off[k] = tot;
    tot += L[k];
  }
  db->total_cols = tot;
  cudaError_t e;
  if ((e = db->cols.alloc((size_t)tot * 7)) != cudaSuccess || (e = db->dL.alloc(n)) != cudaSuccess ||
      (e = db->dcol_off.alloc(n)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_db_create: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->dL.p, db->L.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->dcol_off.p, db->col_off.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  int rc = pack_profiles(ctx, n, L, p_off, tr_off, ss_off, p, tr, ss, db->col_off, tot, db->cols.p);
  if (rc != HHG_OK) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  *out = holder.release();
  return HHG_OK;
}

int hhg_db_create_raw(hhg_ctx* ctx, int n, const int32_t* L, const int64_t* p_off, const int64_t* tr_off,
                      const int64_t* ss_off, const float* p, const float* tr, const uint8_t* ss,
                      const float* pav, hhg_db** out) {
  if (!pav) return fail(HHG_EINVAL, "hhg_db_create_raw: pav is NULL");
  int rc = hhg_db_create(ctx, n, L, p_off, tr_off, ss_off, p, tr, ss, out);
  if (rc != HHG_OK) return rc;
  std::unique_ptr<hhg_db> holder(*out);
  *out = nullptr;
  hhg_db* db = holder.get();
  cudaError_t e;
  if ((e = db->cols_raw.alloc(db->cols.n)) != cudaSuccess || (e = db->pav.alloc((size_t)n * 20)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_db_create_raw: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->cols_raw.p, db->cols.p, db->cols.n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->pav.p, pav, (size_t)n * 20 * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  db->raw = true;
  db->prepared = false;
  *out = holder.release();
  return HHG_OK;
}

int hhg_db_apply_null_model(hhg_ctx* ctx, hhg_db* db, const float* q_pav, const float* pb, int columnscore) {
  if (!ctx || !db || !db->raw) return fail(HHG_EINVAL, "hhg_db_apply_null_model: db was not created raw");
  if (columnscore < 0 || columnscore > 3) return fail(HHG_EINVAL, "columnscore %d not supported (0..3)", columnscore);
  if ((columnscore == 1 || columnscore == 3) && !q_pav) return fail(HHG_EINVAL, "q_pav is NULL");
  if (columnscore == 0 && !pb) return fail(HHG_EINVAL, "pb is NULL");
  CK(cudaSetDevice(ctx->device));
  DevBuf<float> dq;
  CK(dq.alloc(40));
  float h[40] = {0};
  if (q_pav) memcpy(h, q_pav, 80);
  if (pb) memcpy(h + 20, pb, 80);
  CK(cudaMemcpyAsync(dq.p, h, 160, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = 128;
  k_null_model<<<(unsigned)((db->total_cols + threads - 1) / threads), threads, 0, ctx->stream>>>(
      db->total_cols, db->n, db->dcol_off.p, db->cols_raw.p, db->pav.p, dq.p, dq.p + 20, columnscore,
      db->cols.p);
  ctx->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  db->prepared = true;
  db->cols_version++;
  return HHG_OK;
}

// ------------------------------------------------------------------------------ DB from HHM text records
// HHEntry::getTemplateHMM + the query-independent part of PrepareTemplateHMM, once per database load.
// ---------------------------------------------------------------------------------------------------------------
// A3M alignments -> HMMs (hhg_msa.cuh).  One chunk of parsed alignments goes through filter, weights, M state and
// finish; the callers either export the raw HMM (hhg_msa_to_hmm) or continue into the pseudocount step and the shard.
}  // extern "C"
namespace {

struct MsaChunk {
  std::vector<MsaHost> host;
  std::vector<MsaDesc> desc;
  long long seq_total = 0, col_total = 0, x_total = 0, ins_total = 0;
  int Lmax = 0, Nmax = 0;
  DevBuf<MsaDesc> d_desc;
  DevBuf<uint8_t> X, member;
  DevBuf<int8_t> keep, display;
  DevBuf<int> first, last, nres, ksort, in_, inkk, seqid_prev, acc, Ncnt, Nmaxv, idw, ins_k, nfil, status, ni, counter, cnt;
  DevBuf<uint16_t> ins_cnt;
  DevBuf<uint32_t> ins_off;
  DevBuf<float> wg, f, tr, nm, ni_f, nd, nseg, nhmm, wc, wi, pb;
  DevBuf<long long> item_off;
  MsaArrays A{};
};

const float* msa_rcp_table(hhg_ctx* ctx) {
  // RCPPS of this host for every integer argument the weighting can produce (src/hhalignment.cpp:2531)
  static std::vector<float> table;
  static std::once_flag once;
  std::call_once(once, [] {
    table.resize(MSA_RCP_N);
#if defined(__SSE__)
    for (int m = 0; m < MSA_RCP_N; m += 4) {
      const __m128 v = _mm_set_ps((float)(m + 3), (float)(m + 2), (float)(m + 1), (float)m);
      _mm_storeu_ps(&table[m], _mm_rcp_ps(v));
    }
#else
    // no RCPPS on this host: the reference is built through SIMDe there, whose reciprocal estimate differs again;
    // the exact quotient keeps the result well defined (it will not be bit-identical to such a reference build)
    for (int m = 0; m < MSA_RCP_N; ++m) table[m] = 1.0f / (float)m;
#endif
  });
  if (!ctx->msa_rcp) {
    auto buf = std::make_shared<DevBuf<float>>();
    if (buf->alloc(MSA_RCP_N) != cudaSuccess) return nullptr;
    if (cudaMemcpyAsync(buf->p, table.data(), (size_t)MSA_RCP_N * 4, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) return nullptr;
    ctx->msa_rcp = buf;
  }
  return std::static_pointer_cast<DevBuf<float>>(ctx->msa_rcp)->p;
}

#define MSA_CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(HHG_ECUDA, "%s: %s", #x, cudaGetErrorString(e_)); } while (0)

template <typename T, typename V>
int msa_upload(hhg_ctx* ctx, DevBuf<T>& d, const std::vector<V>& h) {
  static_assert(sizeof(T) == sizeof(V), "element size");
  MSA_CK(d.ensure(h.size() ? h.size() : 1));
  if (!h.empty()) MSA_CK(cudaMemcpyAsync(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return HHG_OK;
}

// C.host is filled (parsed); runs the four kernels and leaves f / tr / Neff / keep / wg on the device.
int msa_chunk_run(hhg_ctx* ctx, MsaChunk& C, const hhg_msa_params& mp, const float* S, const float* pb, int first_record) {
  const int m = (int)C.host.size();
  C.desc.resize(m);
  C.seq_total = C.col_total = C.x_total = C.ins_total = 0;
  C.Lmax = C.Nmax = 0;
  std::vector<long long> item_off(m);
  long long items = 0;
  for (int k = 0; k < m; ++k) {
    const MsaHost& H = C.host[k];
    MsaDesc& d = C.desc[k];
    d.N = H.N_in; d.L = H.L; d.stride = H.stride; d.kfirst = H.kfirst;
    d.x_off = C.x_total; d.seq_off = C.seq_total; d.col_off = C.col_total; d.ins_base = C.ins_total;
    C.x_total += (long long)H.N_in * H.stride;
    C.seq_total += H.N_in;
    C.col_total += H.L + 2;
    C.ins_total += (long long)H.ins_k.size();
    C.Lmax = std::max(C.Lmax, H.L); C.Nmax = std::max(C.Nmax, H.N_in);
    item_off[k] = items;
    items += H.L;
  }
  std::vector<uint8_t> X((size_t)C.x_total);
  std::vector<int8_t> keep((size_t)C.seq_total), display((size_t)C.seq_total);
  std::vector<int> first((size_t)C.seq_total), last((size_t)C.seq_total), nres((size_t)C.seq_total), ksort((size_t)C.seq_total);
  std::vector<uint32_t> ins_off((size_t)C.col_total);
  std::vector<int> ins_k((size_t)C.ins_total);
  std::vector<uint16_t> ins_cnt((size_t)C.ins_total);
  for (int k = 0; k < m; ++k) {
    const MsaHost& H = C.host[k];
    const MsaDesc& d = C.desc[k];
    memcpy(X.data() + d.x_off, H.X.data(), H.X.size());
    memcpy(keep.data() + d.seq_off, H.keep.data(), H.N_in);
    memcpy(display.data() + d.seq_off, H.display.data(), H.N_in);
    memcpy(first.data() + d.seq_off, H.first.data(), (size_t)H.N_in * 4);
    memcpy(last.data() + d.seq_off, H.last.data(), (size_t)H.N_in * 4);
    memcpy(nres.data() + d.seq_off, H.nres.data(), (size_t)H.N_in * 4);
    memcpy(ksort.data() + d.seq_off, H.ksort.data(), (size_t)H.N_in * 4);
    memcpy(ins_off.data() + d.col_off, H.ins_off.data(), (size_t)(H.L + 2) * 4);
    if (!H.ins_k.empty()) {
      memcpy(ins_k.data() + d.ins_base, H.ins_k.data(), H.ins_k.size() * 4);
      memcpy(ins_cnt.data() + d.ins_base, H.ins_cnt.data(), H.ins_cnt.size() * 2);
    }
  }
  int rc;
  if ((rc = msa_upload(ctx, C.d_desc, C.desc)) || (rc = msa_upload(ctx, C.X, X)) || (rc = msa_upload(ctx, C.keep, keep)) ||
      (rc = msa_upload(ctx, C.display, display)) || (rc = msa_upload(ctx, C.first, first)) || (rc = msa_upload(ctx, C.last, last)) ||
      (rc = msa_upload(ctx, C.nres, nres)) || (rc = msa_upload(ctx, C.ksort, ksort)) || (rc = msa_upload(ctx, C.ins_off, ins_off)) ||
      (rc = msa_upload(ctx, C.ins_k, ins_k)) || (rc = msa_upload(ctx, C.ins_cnt, ins_cnt)) || (rc = msa_upload(ctx, C.item_off, item_off)))
    return rc;
  const size_t ns = (size_t)C.seq_total, nc = (size_t)C.col_total;
  MSA_CK(C.in_.ensure(ns)); MSA_CK(C.inkk.ensure(ns)); MSA_CK(C.seqid_prev.ensure(ns)); MSA_CK(C.acc.ensure(ns)); MSA_CK(C.wg.ensure(ns));
  MSA_CK(C.Ncnt.ensure(nc)); MSA_CK(C.Nmaxv.ensure(nc)); MSA_CK(C.idw.ensure(nc)); MSA_CK(C.ni.ensure(nc * 21));
  MSA_CK(C.f.ensure(nc * 20)); MSA_CK(C.tr.ensure(nc * 7)); MSA_CK(C.nm.ensure(nc)); MSA_CK(C.ni_f.ensure(nc)); MSA_CK(C.nd.ensure(nc));
  MSA_CK(C.nseg.ensure(nc)); MSA_CK(C.nhmm.ensure(m)); MSA_CK(C.nfil.ensure(m)); MSA_CK(C.status.ensure(m)); MSA_CK(C.counter.ensure(1));
  MSA_CK(C.pb.ensure(20));
  MSA_CK(cudaMemcpyAsync(C.pb.p, pb, 80, cudaMemcpyHostToDevice, ctx->stream));
  MSA_CK(cudaMemsetAsync(C.status.p, 0, (size_t)m * 4, ctx->stream));
  MSA_CK(cudaMemsetAsync(C.counter.p, 0, 4, ctx->stream));
  MSA_CK(cudaMemsetAsync(C.nseg.p, 0, nc * 4, ctx->stream));
  MSA_CK(cudaMemsetAsync(C.tr.p, 0, nc * 7 * 4, ctx->stream));
  const float* rcp = msa_rcp_table(ctx);
  if (!rcp) return fail(HHG_ECUDA, "reciprocal table upload failed");
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  // k_msa_mstate is latency bound inside a block (ordered sums, barriers): 12 blocks of 128 threads per SM = its register /
  // shared-memory residency (40 registers, 16 KB), every block pulls (alignment, column) items until the queue is empty
  const int nblk = (int)std::min<long long>((long long)sms * 12, std::max<long long>(items, 1));
  MSA_CK(C.cnt.ensure((size_t)nblk * (C.Lmax + 2) * 24)); MSA_CK(C.wc.ensure((size_t)nblk * (C.Lmax + 2) * 24));
  MSA_CK(C.wi.ensure((size_t)nblk * C.Nmax)); MSA_CK(C.member.ensure((size_t)nblk * C.Nmax));

  MsaArrays& A = C.A;
  A.desc = C.d_desc.p; A.X = C.X.p; A.keep = C.keep.p; A.display = C.display.p;
  A.first = C.first.p; A.last = C.last.p; A.nres = C.nres.p; A.ksort = C.ksort.p;
  A.in_ = C.in_.p; A.inkk = C.inkk.p; A.seqid_prev = C.seqid_prev.p; A.acc = C.acc.p;
  A.Ncnt = C.Ncnt.p; A.Nmax = C.Nmaxv.p; A.idmaxwin = C.idw.p; A.wg = C.wg.p;
  A.ins_off = C.ins_off.p; A.ins_k = C.ins_k.p; A.ins_cnt = C.ins_cnt.p;
  A.n_filtered = C.nfil.p; A.status = C.status.p;
  A.f = C.f.p; A.tr = C.tr.p; A.neff_m = C.nm.p; A.neff_i = C.ni_f.p; A.neff_d = C.nd.p; A.neff_seg = C.nseg.p; A.neff_hmm = C.nhmm.p;

  MsaFilterParams FP;
  FP.max_seqid = mp.max_seqid; FP.coverage = mp.coverage; FP.qid = mp.qid; FP.Ndiff = mp.Ndiff; FP.qsc = mp.qsc;
  if (S) memcpy(FP.S, S, sizeof(FP.S)); else memset(FP.S, 0, sizeof(FP.S));
  const bool timing = getenv("HHG_TIMING") != nullptr;
  cudaEvent_t ev[5] = {};
  if (timing) for (auto& e : ev) cudaEventCreate(&e);
  if (timing) cudaEventRecord(ev[0], ctx->stream);
  k_msa_filter<<<m, 256, 0, ctx->stream>>>(A, FP);
  if (timing) cudaEventRecord(ev[1], ctx->stream);
  k_msa_weights<<<m, 256, 0, ctx->stream>>>(A, C.ni.p);
  if (timing) cudaEventRecord(ev[2], ctx->stream);
  k_msa_mstate<<<nblk, MSA_MSTATE_THREADS, 0, ctx->stream>>>(A, m, C.item_off.p, items, C.counter.p, C.cnt.p, C.wc.p, C.wi.p, C.member.p,
                                              C.Lmax, C.Nmax, rcp, C.pb.p, mp.wg ? 1 : 0, ctx->lg2.p, ctx->diff.p);
  if (timing) cudaEventRecord(ev[3], ctx->stream);
  k_msa_finish<<<m, 256, 0, ctx->stream>>>(A, C.pb.p, mp.wg ? 1 : 0, ctx->lg2.p, ctx->diff.p);
  if (timing) cudaEventRecord(ev[4], ctx->stream);
  ctx->launches += 4;
  MSA_CK(cudaGetLastError());
  if (timing) {
    cudaEventSynchronize(ev[4]);
    float t[4];
    for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&t[k], ev[k], ev[k + 1]);
    fprintf(stderr, "[hhg] alignment kernels (%d alignments, %lld columns): filter %.2f ms, weights %.2f ms, M state %.2f ms, finish %.2f ms\n",
            m, items, t[0], t[1], t[2], t[3]);
    for (auto& e : ev) cudaEventDestroy(e);
  }
  std::vector<int> status(m);
  MSA_CK(cudaMemcpyAsync(status.data(), C.status.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
  MSA_CK(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < m; ++k)
    if (status[k])
      return fail(HHG_EINVAL, "alignment %d: %s", first_record + k,
                  status[k] == 1 ? "contains no sequences after filtering (the reference exits here)"
                  : status[k] == 2 ? "the position-dependent identity schedule divides by zero (as in the reference)"
                                   : "no sequence left for the profile");
  return HHG_OK;
}

int msa_params_check(const hhg_msa_params* mp) {
  if (!mp) return fail(HHG_EINVAL, "alignment parameters are NULL");
  if (mp->maxseq < 2 || mp->maxseq > 65535) return fail(HHG_EINVAL, "maxseq %d outside [2, 65535]", mp->maxseq);
  if (mp->maxres < 8 || mp->maxcol < mp->maxres) return fail(HHG_EINVAL, "maxres %d / maxcol %d", mp->maxres, mp->maxcol);
  if (mp->M < 1 || mp->M > 3) return fail(HHG_EINVAL, "match-state assignment %d: 1 (A2M/A3M: upper case = match), 2 (gap percentage, Mgaps) or 3 (first sequence)", mp->M);
  if (mp->M == 2 && (mp->Mgaps < 0 || mp->Mgaps > 100)) return fail(HHG_EINVAL, "Mgaps %d outside [0, 100]", mp->Mgaps);
  if (mp->mark != 0) return fail(HHG_EINVAL, "the -mark option is not built");
  return HHG_OK;
}

// ss byte of column j (1..L) the DP reads: ss_pred * MAXCF + ss_conf (src/hhhmmsimd.cpp:133); ss_conf = 5 without an
// ss_conf row (FrequenciesAndTransitions :2313-2319)
void msa_ss_bytes(const MsaHost& H, uint8_t* out) {
  if (H.kss_pred < 0) { memset(out, 0, (size_t)H.L); return; }
  const uint8_t* pr = H.X.data() + (size_t)H.kss_pred * H.stride;
  const uint8_t* cf = H.kss_conf >= 0 ? H.X.data() + (size_t)H.kss_conf * H.stride : nullptr;
  for (int j = 1; j <= H.L; ++j) out[j - 1] = (uint8_t)((pr[j] & 0x7f) * 11 + (cf ? (cf[j] & 0x7f) : 5));
}

}  // namespace
extern "C" {

void hhg_msa_params_default(hhg_msa_params* mp) {
  if (!mp) return;
  mp->maxseq = 65535; mp->maxcol = 32765; mp->maxres = 20001;       // src/hhdecl.cpp:10-14
  mp->M = 1; mp->mark = 0;
  mp->max_seqid = 90; mp->coverage = 0; mp->qid = 0; mp->Ndiff = 100; mp->qsc = -20.0f;   // :35-39, :131-135
  mp->wg = 0;
  mp->Mgaps = 50;                                                    // :46
}

int hhg_a3m_scan(const char* rec, int64_t len, const hhg_msa_params* mp, int32_t* L, int32_t* N_in, int32_t* has_ss) {
  if (!rec || len <= 0 || !L || !N_in) return fail(HHG_EINVAL, "hhg_a3m_scan: bad argument");
  int rc = msa_params_check(mp);
  if (rc != HHG_OK) return rc;
  MsaHost H;
  const std::string msg = MsaScanner::parse(rec, len, mp->maxseq, mp->maxcol, mp->maxres, &H, mp->M, mp->Mgaps);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_a3m_scan: %s", msg.c_str());
  *L = H.L; *N_in = H.N_in;
  if (has_ss) *has_ss = H.kss_pred >= 0;
  return HHG_OK;
}

static int seqdb_check(const hhg_seqdb* sq) {
  if (!sq) return HHG_OK;
  if (sq->n <= 0 || !sq->data || !sq->off || !sq->len) return fail(HHG_EINVAL, "sequence database: bad argument");
  return HHG_OK;
}

static std::string msa_parse_any(const char* rec, int64_t len, const hhg_seqdb* sq, const hhg_msa_params* mp, MsaHost* H) {
  if (!sq) return MsaScanner::parse(rec, len, mp->maxseq, mp->maxcol, mp->maxres, H, mp->M, mp->Mgaps);
  const MsaScanner::SeqDb db{sq->n, sq->data, sq->off, sq->len};
  return MsaScanner::parse_ca3m(rec, len, db, mp->maxseq, mp->maxcol, mp->maxres, H, mp->M, mp->Mgaps);
}

static int msa_parse_impl(const char* rec, int64_t len, const hhg_seqdb* sq, const hhg_msa_params* mp, int32_t L_cap,
                          int32_t N_cap, int32_t* dims, uint8_t* X, uint16_t* I, int8_t* keep, int32_t* nres, int32_t* ksort) {
  if (!rec || len <= 0 || !dims || !X) return fail(HHG_EINVAL, "hhg_a3m_parse: bad argument");
  int rc = msa_params_check(mp);
  if (rc != HHG_OK) return rc;
  if ((rc = seqdb_check(sq)) != HHG_OK) return rc;
  MsaHost H;
  const std::string msg = msa_parse_any(rec, len, sq, mp, &H);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_a3m_parse: %s", msg.c_str());
  dims[0] = H.L; dims[1] = H.N_in; dims[2] = 0; dims[3] = H.kfirst; dims[4] = H.kss_pred; dims[5] = H.kss_conf;
  if (H.L > L_cap || H.N_in > N_cap) return fail(HHG_EINVAL, "hhg_a3m_parse: %d columns / %d sequences exceed the caller's capacity", H.L, H.N_in);
  const int L = H.L, N = H.N_in;
  for (int k = 0; k < N; ++k) {
    for (int i = 0; i <= L + 1; ++i) X[(size_t)k * (L + 2) + i] = H.X[(size_t)k * H.stride + i] & 0x7f;
    if (I) for (int i = 0; i <= L + 1; ++i) I[(size_t)k * (L + 2) + i] = 0;
    if (keep) keep[k] = H.keep[k];
    if (nres) nres[k] = H.nres[k];
    if (ksort) ksort[k] = H.ksort[k];
  }
  if (I)
    for (int i = 0; i <= L; ++i)
      for (uint32_t e = H.ins_off[i]; e < H.ins_off[i + 1]; ++e) I[(size_t)H.ins_k[e] * (L + 2) + i] = H.ins_cnt[e];
  return HHG_OK;
}

int hhg_a3m_parse(const char* rec, int64_t len, const hhg_msa_params* mp, int32_t L_cap, int32_t N_cap, int32_t* dims,
                  uint8_t* X, uint16_t* I, int8_t* keep, int32_t* nres, int32_t* ksort) {
  return msa_parse_impl(rec, len, nullptr, mp, L_cap, N_cap, dims, X, I, keep, nres, ksort);
}

int hhg_ca3m_parse(const char* rec, int64_t len, const hhg_seqdb* seqs, const hhg_msa_params* mp, int32_t L_cap, int32_t N_cap,
                   int32_t* dims, uint8_t* X, uint16_t* I, int8_t* keep, int32_t* nres, int32_t* ksort) {
  if (!seqs) return fail(HHG_EINVAL, "hhg_ca3m_parse: the sequence database is NULL");
  return msa_parse_impl(rec, len, seqs, mp, L_cap, N_cap, dims, X, I, keep, nres, ksort);
}

static int msa_to_hmm_impl(hhg_ctx* ctx, const char* rec, int64_t len, const hhg_seqdb* sq, const hhg_msa_params* mp,
                           const float* S, const float* pb, int32_t L_cap, int32_t N_cap, int32_t* dims, int8_t* keep,
                           float* wg, float* f, float* tr, float* neff, float* neff_hmm, uint8_t* ss) {
  if (!ctx || !rec || len <= 0 || !pb || !dims || !f || !tr || !neff || !neff_hmm)
    return fail(HHG_EINVAL, "hhg_msa_to_hmm: bad argument");
  int rc = msa_params_check(mp);
  if (rc != HHG_OK) return rc;
  if ((rc = seqdb_check(sq)) != HHG_OK) return rc;
  if (mp->qsc > -10.f && !S) return fail(HHG_EINVAL, "hhg_msa_to_hmm: the qsc filter needs the substitution matrix S");
  CK(cudaSetDevice(ctx->device));
  if (!ctx->msa_cache) ctx->msa_cache = std::make_shared<MsaChunk>();      // device buffers persist between calls
  MsaChunk& C = *std::static_pointer_cast<MsaChunk>(ctx->msa_cache);
  C.host.clear();
  C.host.resize(1);
  const std::string msg = msa_parse_any(rec, len, sq, mp, &C.host[0]);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_msa_to_hmm: %s", msg.c_str());
  const MsaHost& H = C.host[0];
  dims[0] = H.L; dims[1] = H.N_in; dims[2] = 0; dims[3] = H.kfirst; dims[4] = H.kss_pred; dims[5] = H.kss_conf;
  if (H.L > L_cap || H.N_in > N_cap) return fail(HHG_EINVAL, "hhg_msa_to_hmm: %d columns / %d sequences exceed the caller's capacity %d / %d", H.L, H.N_in, L_cap, N_cap);
  rc = msa_chunk_run(ctx, C, *mp, S, pb, 0);
  if (rc != HHG_OK) return rc;
  const int L = H.L, N = H.N_in;
  int nf = 0;
  CK(cudaMemcpyAsync(&nf, C.nfil.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (keep) CK(cudaMemcpyAsync(keep, C.keep.p, (size_t)N, cudaMemcpyDeviceToHost, ctx->stream));
  if (wg) CK(cudaMemcpyAsync(wg, C.wg.p, (size_t)N * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(f, C.f.p, (size_t)(L + 2) * 80, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(tr, C.tr.p, (size_t)(L + 1) * 28, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(neff, C.nm.p, (size_t)(L + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(neff + (L + 1), C.ni_f.p, (size_t)(L + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(neff + 2 * (L + 1), C.nd.p, (size_t)(L + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(neff_hmm, C.nhmm.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  dims[2] = nf;
  if (ss) { ss[0] = 0; msa_ss_bytes(H, ss + 1); ss[L + 1] = 0; }
  return HHG_OK;
}

int hhg_msa_to_hmm(hhg_ctx* ctx, const char* rec, int64_t len, const hhg_msa_params* mp, const float* S, const float* pb,
                   int32_t L_cap, int32_t N_cap, int32_t* dims, int8_t* keep, float* wg, float* f, float* tr,
                   float* neff, float* neff_hmm, uint8_t* ss) {
  return msa_to_hmm_impl(ctx, rec, len, nullptr, mp, S, pb, L_cap, N_cap, dims, keep, wg, f, tr, neff, neff_hmm, ss);
}

int hhg_ca3m_to_hmm(hhg_ctx* ctx, const char* rec, int64_t len, const hhg_seqdb* seqs, const hhg_msa_params* mp,
                    const float* S, const float* pb, int32_t L_cap, int32_t N_cap, int32_t* dims, int8_t* keep, float* wg,
                    float* f, float* tr, float* neff, float* neff_hmm) {
  if (!seqs) return fail(HHG_EINVAL, "hhg_ca3m_to_hmm: the sequence database is NULL");
  return msa_to_hmm_impl(ctx, rec, len, seqs, mp, S, pb, L_cap, N_cap, dims, keep, wg, f, tr, neff, neff_hmm, nullptr);
}

int hhg_ca3m_scan(const char* rec, int64_t len, const hhg_seqdb* seqs, const hhg_msa_params* mp, int32_t* L, int32_t* N_in) {
  if (!rec || len <= 0 || !L || !N_in || !seqs) return fail(HHG_EINVAL, "hhg_ca3m_scan: bad argument");
  int rc = msa_params_check(mp);
  if (rc != HHG_OK) return rc;
  if ((rc = seqdb_check(seqs)) != HHG_OK) return rc;
  MsaHost H;
  const std::string msg = msa_parse_any(rec, len, seqs, mp, &H);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_ca3m_scan: %s", msg.c_str());
  *L = H.L; *N_in = H.N_in;
  return HHG_OK;
}

static int db_create_a3m_impl(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len,
                              const hhg_seqdb* sq, const hhg_msa_params* mp, const float* S, const float* pb,
                              const hhg_prep_params* pp, const float* R, hhg_db** out, float* d_tr_full,
                              float* neff_hmm_out) {
  if (!ctx || !out || n <= 0 || !data || !off || !len || !pp || !R || !pb)
    return fail(HHG_EINVAL, "hhg_db_create_a3m: bad argument");
  int rc = msa_params_check(mp);
  if (rc != HHG_OK) return rc;
  if ((rc = seqdb_check(sq)) != HHG_OK) return rc;
  if (mp->qsc > -10.f && !S) return fail(HHG_EINVAL, "hhg_db_create_a3m: the qsc filter needs the substitution matrix S");
  if (pp->pcm < 0 || pp->pcm > 3) return fail(HHG_EINVAL, "hhg_db_create_a3m: pseudocount mode %d does not exist", pp->pcm);
  const bool tau_on_host = pp->pcm == 2 && pp->pcc != 1.0f;
  CK(cudaSetDevice(ctx->device));
  const bool timing = getenv("HHG_TIMING") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  double ms_scan = 0.0, ms_kernels = 0.0;

  HhmPrepArgs A;
  memcpy(A.R, R, sizeof(A.R));
  A.gapb = pp->gapb; A.gapf = pp->gapf; A.gapg = pp->gapg; A.gaph = pp->gaph; A.gapi = pp->gapi;
  A.pM2D = A.pM2I = (float)(pp->gapd * 0.0286);
  A.pM2M = 1 - A.pM2D - A.pM2I;
  A.pI2I = (float)(1.0 * pp->gape / (pp->gape - 1 + 1.0 / 0.75));
  A.pI2M = 1 - A.pI2I;
  A.pD2D = (float)(1.0 * pp->gape / (pp->gape - 1 + 1.0 / 0.75));
  A.pD2M = 1 - A.pD2D;
  A.pcm = pp->pcm; A.pca = pp->pca; A.pcb = pp->pcb; A.pcc = pp->pcc;

  // The records go through in groups: host scan of a group (threads) -> kernels -> column records of the group in a
  // device piece; the shard is assembled from the pieces at the end.  Host memory holds one group of parsed
  // alignments at a time (a database of alignments is far larger than the shard it turns into).
  struct Piece { DevBuf<float4> cols; DevBuf<float> pav; int first = 0, n = 0; long long ncols = 0; };
  std::vector<std::unique_ptr<Piece>> pieces;
  std::unique_ptr<hhg_db> holder(new hhg_db());
  hhg_db* db = holder.get();
  db->device = ctx->device;
  db->n = n;
  db->L.resize(n);
  db->col_off.resize(n);
  long long tot = 0;
  bool any_ss = false;

  const long long kGroupText = 256ll << 20;           // bytes of input text per group
  int max_records = 8192;
  { const char* e = getenv("HHG_MSA_CHUNK_RECORDS"); if (e && atoi(e) > 0) max_records = atoi(e); }   // test knob: many small groups
  MsaChunk C;
  DevBuf<long long> d_rec_off;
  DevBuf<uint8_t> d_ss;
  DevBuf<float> d_tau;
  DevBuf<int> d_L;
  const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  int t0 = 0;
  while (t0 < n) {
    int t1 = t0;
    long long bytes = 0;
    while (t1 < n && t1 - t0 < max_records && (bytes == 0 || bytes + len[t1] <= kGroupText)) bytes += len[t1++];
    const int m = t1 - t0;
    const auto t_s0 = std::chrono::steady_clock::now();
    C.host.clear();
    C.host.resize(m);
    {
      std::vector<std::string> errs(hw);
      std::vector<int> err_rec(hw, -1);
      auto work = [&](unsigned w) {
        for (int k = (int)w; k < m; k += (int)hw) {
          if (len[t0 + k] <= 0) { if (err_rec[w] < 0) { errs[w] = "empty record"; err_rec[w] = t0 + k; } continue; }
          std::string msg = msa_parse_any(data + off[t0 + k], len[t0 + k], sq, mp, &C.host[k]);
          if (!msg.empty() && err_rec[w] < 0) { errs[w] = msg; err_rec[w] = t0 + k; }
        }
      };
      std::vector<std::thread> pool;
      for (unsigned w = 1; w < hw; ++w) pool.emplace_back(work, w);
      work(0);
      for (auto& th : pool) th.join();
      for (unsigned w = 0; w < hw; ++w)
        if (err_rec[w] >= 0) return fail(HHG_EINVAL, "record %d: %s", err_rec[w], errs[w].c_str());
    }
    std::vector<long long> rec_off(m);
    std::vector<int> Lg(m);
    long long cols = 0;
    for (int k = 0; k < m; ++k) {
      const int L = C.host[k].L;
      if (L > 32767) return fail(HHG_EINVAL, "record %d: length %d out of [1,32767]", t0 + k, L);
      db->L[t0 + k] = L; db->col_off[t0 + k] = tot + cols;
      rec_off[k] = cols; Lg[k] = L; cols += L;
      any_ss |= C.host[k].kss_pred >= 0;
    }
    ms_scan += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_s0).count();
    const auto t_c0 = std::chrono::steady_clock::now();
    rc = msa_chunk_run(ctx, C, *mp, S, pb, t0);
    if (rc != HHG_OK) return rc;
    ms_kernels += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_c0).count();
    std::vector<uint8_t> ssb((size_t)cols, 0);
    for (int k = 0; k < m; ++k) msa_ss_bytes(C.host[k], ssb.data() + rec_off[k]);
    CK(d_rec_off.ensure(m)); CK(d_ss.ensure((size_t)cols)); CK(d_L.ensure(m));
    CK(cudaMemcpyAsync(d_rec_off.p, rec_off.data(), (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_ss.p, ssb.data(), (size_t)cols, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_L.p, Lg.data(), (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
    std::vector<float> tau_h;
    if (tau_on_host) {
      std::vector<float> nm((size_t)C.col_total);
      CK(cudaMemcpyAsync(nm.data(), C.nm.p, nm.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      tau_h.resize((size_t)cols);
      for (int k = 0; k < m; ++k)
        for (int j = 1; j <= C.host[k].L; ++j)
          tau_h[(size_t)rec_off[k] + j - 1] = (float)fmin(1.0, pp->pca / (1. + powf(nm[(size_t)C.desc[k].col_off + j] / pp->pcb, pp->pcc)));
      CK(d_tau.ensure((size_t)cols));
      CK(cudaMemcpyAsync(d_tau.p, tau_h.data(), (size_t)cols * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    pieces.emplace_back(new Piece());
    Piece& P = *pieces.back();
    P.first = t0; P.n = m; P.ncols = cols;
    cudaError_t e;
    if ((e = P.cols.alloc((size_t)cols * 7)) != cudaSuccess || (e = P.pav.alloc((size_t)m * 20)) != cudaSuccess)
      return fail(HHG_ENOMEM, "hhg_db_create_a3m: %s", cudaGetErrorString(e));
    ColRec* dst = reinterpret_cast<ColRec*>(P.cols.p);
    const int threads = 128;
    k_msa_prepare<<<(unsigned)((cols + threads - 1) / threads), threads, 0, ctx->stream>>>(
        m, C.d_desc.p, d_rec_off.p, C.A, d_ss.p, A, ctx->lg2.p, ctx->diff.p, dst, cols, d_tr_full,
        tau_on_host ? d_tau.p : nullptr);
    k_hhm_pav<<<(unsigned)(((long long)m * 32 + threads - 1) / threads), threads, 0, ctx->stream>>>(
        m, d_L.p, d_rec_off.p, dst, nullptr, C.nhmm.p, A, P.pav.p, C.pb.p);
    ctx->launches += 2;
    CK(cudaGetLastError());
    if (neff_hmm_out) CK(cudaMemcpyAsync(neff_hmm_out + t0, C.nhmm.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));     // host staging of the group is reused by the next one
    tot += cols;
    t0 = t1;
  }
  db->total_cols = tot;
  db->has_ss = any_ss;
  cudaError_t e;
  if ((e = db->cols.alloc((size_t)tot * 7)) != cudaSuccess || (e = db->cols_raw.alloc((size_t)tot * 7)) != cudaSuccess ||
      (e = db->dL.alloc(n)) != cudaSuccess || (e = db->dcol_off.alloc(n)) != cudaSuccess ||
      (e = db->pav.alloc((size_t)n * 20)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_db_create_a3m: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->dL.p, db->L.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->dcol_off.p, db->col_off.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  long long at = 0;
  for (auto& pc : pieces) {
    CK(cudaMemcpyAsync(db->cols_raw.p + (size_t)at * 7, pc->cols.p, (size_t)pc->ncols * 7 * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemcpyAsync(db->pav.p + (size_t)pc->first * 20, pc->pav.p, (size_t)pc->n * 80, cudaMemcpyDeviceToDevice, ctx->stream));
    at += pc->ncols;
  }
  CK(cudaMemcpyAsync(db->cols.p, db->cols_raw.p, db->cols.n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  pieces.clear();
  if (timing) {
    const double ms_all = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    fprintf(stderr, "[hhg] alignment loader: %d records, host scan %.1f ms, staging + filter/weights/M-state/finish kernels %.1f ms, "
                    "rest (pseudocounts, pav, copies) %.1f ms\n", n, ms_scan, ms_kernels, ms_all - ms_scan - ms_kernels);
  }
  db->raw = true;
  db->prepared = false;
  *out = holder.release();
  return HHG_OK;
}

int hhg_db_create_a3m(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len,
                      const hhg_msa_params* mp, const float* S, const float* pb, const hhg_prep_params* pp,
                      const float* R, hhg_db** out) {
  return db_create_a3m_impl(ctx, n, data, off, len, nullptr, mp, S, pb, pp, R, out, nullptr, nullptr);
}

int hhg_db_create_ca3m(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len, const hhg_seqdb* seqs,
                       const hhg_msa_params* mp, const float* S, const float* pb, const hhg_prep_params* pp,
                       const float* R, hhg_db** out) {
  if (!seqs) return fail(HHG_EINVAL, "hhg_db_create_ca3m: the sequence database is NULL");
  return db_create_a3m_impl(ctx, n, data, off, len, seqs, mp, S, pb, pp, R, out, nullptr, nullptr);
}

int hhg_hhm_scan(const char* rec, int64_t len, int32_t* L, int32_t* has_ss) {
  if (!rec || len <= 0 || !L || !has_ss) return fail(HHG_EINVAL, "hhg_hhm_scan: bad argument");
  HhmScanner sc(rec, len);
  if (!sc.peek(L, has_ss)) return fail(HHG_EINVAL, "hhg_hhm_scan: no LENG line / not an HHM record");
  return HHG_OK;
}

int hhg_hhm_parse(const char* rec, int64_t len, int32_t L, int32_t* f_mb, int32_t* trn_mb, uint8_t* ss,
                  int32_t* null_mb, float* neff_hmm, int32_t* has_pc) {
  if (!rec || len <= 0 || L < 1 || !f_mb || !trn_mb || !ss || !null_mb || !neff_hmm || !has_pc)
    return fail(HHG_EINVAL, "hhg_hhm_parse: bad argument");
  HhmScanner sc(rec, len);
  std::string msg = sc.parse(L, f_mb, trn_mb, ss, null_mb, neff_hmm, has_pc);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_hhm_parse: %s", msg.c_str());
  return HHG_OK;
}

static int db_create_hhm_impl(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len,
                              const hhg_prep_params* pp, const float* R, hhg_db** out, float* d_tr_full) {
  if (!ctx || !out || n <= 0 || !data || !off || !len || !pp || !R)
    return fail(HHG_EINVAL, "hhg_db_create_hhm: bad argument");
  if (pp->pcm < 0 || pp->pcm > 3)
    return fail(HHG_EINVAL, "hhg_db_create_hhm: pseudocount mode %d does not exist (src/hhhmm.cpp:1885-1918: 0..3)", pp->pcm);
  const bool tau_on_host = pp->pcm == 2 && pp->pcc != 1.0f;   // needs the C library's powf: computed per column below
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<hhg_db> holder(new hhg_db());
  hhg_db* db = holder.get();
  db->device = ctx->device;
  db->n = n;
  db->L.resize(n);
  db->col_off.resize(n);
  // pass 1: lengths (LENG) and whether any record predicts secondary structure
  long long tot = 0;
  bool any_ss = false;
  for (int k = 0; k < n; ++k) {
    int32_t L = 0, has_ss = 0;
    HhmScanner sc(data + off[k], len[k]);
    if (len[k] <= 0 || !sc.peek(&L, &has_ss)) return fail(HHG_EINVAL, "record %d: no LENG line / not an HHM record", k);
    if (L < 1 || L > 32767) return fail(HHG_EINVAL, "record %d: length %d out of [1,32767]", k, L);
    db->L[k] = L;
    db->col_off[k] = tot;
    tot += L;
    any_ss |= has_ss != 0;
  }
  db->total_cols = tot;
  db->has_ss = any_ss;
  cudaError_t e;
  if ((e = db->cols.alloc((size_t)tot * 7)) != cudaSuccess || (e = db->cols_raw.alloc((size_t)tot * 7)) != cudaSuccess ||
      (e = db->dL.alloc(n)) != cudaSuccess || (e = db->dcol_off.alloc(n)) != cudaSuccess ||
      (e = db->pav.alloc((size_t)n * 20)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_db_create_hhm: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->dL.p, db->L.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->dcol_off.p, db->col_off.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));

  HhmPrepArgs A;
  memcpy(A.R, R, sizeof(A.R));
  A.gapb = pp->gapb; A.gapf = pp->gapf; A.gapg = pp->gapg; A.gaph = pp->gaph; A.gapi = pp->gapi;
  A.pM2D = A.pM2I = (float)(pp->gapd * 0.0286);                       // src/hhhmm.cpp:1745-1752, same types
  A.pM2M = 1 - A.pM2D - A.pM2I;
  A.pI2I = (float)(1.0 * pp->gape / (pp->gape - 1 + 1.0 / 0.75));
  A.pI2M = 1 - A.pI2I;
  A.pD2D = (float)(1.0 * pp->gape / (pp->gape - 1 + 1.0 / 0.75));
  A.pD2M = 1 - A.pD2D;
  A.pcm = pp->pcm; A.pca = pp->pca; A.pcb = pp->pcb; A.pcc = pp->pcc;

  // pass 2: chunks of records -> host staging (parsed by a few threads) -> device -> k_hhm_prepare / k_hhm_pav
  const long long kChunkCols = 2000000;
  DevBuf<int32_t> d_f, d_trn, d_null, d_haspc;
  DevBuf<uint8_t> d_ss;
  DevBuf<float> d_neff, d_tau;
  DevBuf<long long> d_coff;
  std::vector<float> tau_h;
  HhmStaging st;
  std::vector<long long> coff;
  const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  int t0 = 0;
  while (t0 < n) {
    int t1 = t0;
    long long cols = 0;
    while (t1 < n && (cols == 0 || cols + db->L[t1] <= kChunkCols)) cols += db->L[t1++];
    const int m = t1 - t0;
    coff.resize(m);
    for (int k = 0; k < m; ++k) coff[k] = db->col_off[t0 + k] - db->col_off[t0];
    st.f_mb.assign((size_t)cols * 20, 0);
    st.trn_mb.assign((size_t)(cols + m) * 10, 0);
    st.ss.assign((size_t)cols, 0);
    st.null_mb.assign((size_t)m * 20, 0);
    st.neff_hmm.assign(m, 0.f);
    st.has_pc.assign(m, 0);
    std::vector<std::string> errs(hw);
    std::vector<int> err_rec(hw, -1);
    auto work = [&](unsigned w) {
      for (int k = (int)w; k < m; k += (int)hw) {
        HhmScanner sc(data + off[t0 + k], len[t0 + k]);
        std::string msg = sc.parse(db->L[t0 + k], st.f_mb.data() + (size_t)coff[k] * 20,
                                   st.trn_mb.data() + (size_t)(coff[k] + k) * 10, st.ss.data() + coff[k],
                                   st.null_mb.data() + (size_t)k * 20, &st.neff_hmm[k], &st.has_pc[k]);
        if (!msg.empty() && err_rec[w] < 0) { errs[w] = msg; err_rec[w] = t0 + k; }
      }
    };
    std::vector<std::thread> pool;
    for (unsigned w = 1; w < hw; ++w) pool.emplace_back(work, w);
    work(0);
    for (auto& th : pool) th.join();
    for (unsigned w = 0; w < hw; ++w)
      if (err_rec[w] >= 0) return fail(HHG_EINVAL, "record %d: %s", err_rec[w], errs[w].c_str());
    CK(d_f.ensure(st.f_mb.size())); CK(d_trn.ensure(st.trn_mb.size())); CK(d_ss.ensure(st.ss.size()));
    CK(d_null.ensure(st.null_mb.size())); CK(d_haspc.ensure(m)); CK(d_neff.ensure(m)); CK(d_coff.ensure(m));
    CK(cudaMemcpyAsync(d_f.p, st.f_mb.data(), st.f_mb.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_trn.p, st.trn_mb.data(), st.trn_mb.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_ss.p, st.ss.data(), st.ss.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_null.p, st.null_mb.data(), st.null_mb.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_haspc.p, st.has_pc.data(), (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_neff.p, st.neff_hmm.data(), (size_t)m * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_coff.p, coff.data(), (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (tau_on_host) {
      // AddAminoAcidPseudocounts mode 2 with pcc != 1 (src/hhhmm.cpp:1905-1909): tau = fmin(1.0, pca / (1. + pow(Neff_M/pcb, pcc)))
      // with float arguments, i.e. the C library's powf; one value per column, computed here with the same libm
      tau_h.resize((size_t)cols);
      for (int k = 0; k < m; ++k) {
        const int32_t* rows = st.trn_mb.data() + (size_t)(coff[k] + k) * 10;
        for (int j = 1; j <= db->L[t0 + k]; ++j) {
          const float nM = (float)rows[(size_t)j * 10 + 7] / 1000.0f;
          tau_h[(size_t)coff[k] + j - 1] = (float)fmin(1.0, pp->pca / (1. + powf(nM / pp->pcb, pp->pcc)));
        }
      }
      CK(d_tau.ensure((size_t)cols));
      CK(cudaMemcpyAsync(d_tau.p, tau_h.data(), (size_t)cols * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    ColRec* dst = reinterpret_cast<ColRec*>(db->cols_raw.p) + db->col_off[t0];
    const int threads = 128;
    k_hhm_prepare<<<(unsigned)((cols + threads - 1) / threads), threads, 0, ctx->stream>>>(
        m, db->dL.p + t0, d_coff.p, d_f.p, d_trn.p, any_ss ? d_ss.p : nullptr, d_haspc.p, A, ctx->lg2.p,
        ctx->diff.p, dst, cols, d_tr_full,    // d_tr_full only with a single chunk (hhg_query_from_hhm: one record)
        tau_on_host ? d_tau.p : nullptr);
    k_hhm_pav<<<(unsigned)(((long long)m * 32 + threads - 1) / threads), threads, 0, ctx->stream>>>(
        m, db->dL.p + t0, d_coff.p, dst, d_null.p, d_neff.p, A, db->pav.p + (size_t)t0 * 20);
    ctx->launches += 2;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));   // staging is reused by the next chunk
    t0 = t1;
  }
  CK(cudaMemcpyAsync(db->cols.p, db->cols_raw.p, db->cols.n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  db->raw = true;
  db->prepared = false;
  *out = holder.release();
  return HHG_OK;
}

int hhg_db_create_hhm(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len,
                      const hhg_prep_params* pp, const float* R, hhg_db** out) {
  return db_create_hhm_impl(ctx, n, data, off, len, pp, R, out, nullptr);
}

// PrepareQueryHMM for an HHM query without context-specific pseudocounts (par.nocontxt; src/hhfunc.cpp:121-160): the
// same three steps a template gets -- AddTransitionPseudocounts, PreparePseudocounts + AddAminoAcidPseudocounts,
// CalculateAminoAcidBackground -- so the record runs through the database loader's kernels and comes back as the host
// arrays hhg_query_set / hhg_prefilter_build_profile take.
int hhg_query_from_hhm(hhg_ctx* ctx, const char* rec, int64_t len, const hhg_prep_params* pp, const float* R,
                       int32_t L_cap, int32_t* L_out, float* p, float* tr, uint8_t* ss, float* pav, float* neff) {
  if (!ctx || !rec || len <= 0 || !pp || !R || !L_out || !p || !tr || !pav) return fail(HHG_EINVAL, "hhg_query_from_hhm: bad argument");
  int32_t L = 0, has_ss = 0;
  { HhmScanner sc(rec, len); if (!sc.peek(&L, &has_ss)) return fail(HHG_EINVAL, "hhg_query_from_hhm: not an HHM record"); }
  if (L < 1 || L > L_cap) return fail(HHG_EINVAL, "hhg_query_from_hhm: query length %d exceeds the caller's capacity %d", L, L_cap);
  CK(cudaSetDevice(ctx->device));
  DevBuf<float> d_tr;
  CK(d_tr.alloc((size_t)(L + 1) * 7));
  hhg_db* db = nullptr;
  const int64_t zero = 0;
  int rc = db_create_hhm_impl(ctx, 1, rec, &zero, &len, pp, R, &db, d_tr.p);
  if (rc != HHG_OK) return rc;
  std::unique_ptr<hhg_db> holder(db);
  std::vector<ColRec> cols((size_t)L);
  CK(cudaMemcpyAsync(cols.data(), db->cols_raw.p, (size_t)L * sizeof(ColRec), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(tr, d_tr.p, (size_t)(L + 1) * 28, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(pav, db->pav.p, 80, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int i = 1; i <= L; ++i) {
    memcpy(p + (size_t)i * 20, cols[i - 1].p, 80);
    if (ss) ss[i] = (uint8_t)cols[i - 1].ss;
  }
  memcpy(p, pav, 80);                               // CalculateAminoAcidBackground: p[0] = p[L+1] = pav (:1866)
  memcpy(p + (size_t)(L + 1) * 20, pav, 80);
  if (ss) ss[0] = ss[L + 1] = 0;
  if (neff) {
    std::vector<int32_t> f((size_t)L * 20), trn((size_t)(L + 1) * 10), nul(20);
    std::vector<uint8_t> ssb(L);
    int32_t has_pc = 0;
    rc = hhg_hhm_parse(rec, len, L, f.data(), trn.data(), ssb.data(), nul.data(), neff, &has_pc);
    if (rc != HHG_OK) return rc;
  }
  *L_out = L;
  return HHG_OK;
}

// The same for a query ALIGNMENT (hhblits: ReadQueryFile -> Alignment::Read / Compress / Filter /
// FrequenciesAndTransitions, src/hhblits.cpp:1424-1453, then PrepareQueryHMM's nocontxt branch).
int hhg_query_from_a3m(hhg_ctx* ctx, const char* rec, int64_t len, const hhg_msa_params* mp, const float* S, const float* pb,
                       const hhg_prep_params* pp, const float* R, int32_t L_cap, int32_t* L_out, float* p, float* tr,
                       uint8_t* ss, float* pav, float* neff) {
  if (!ctx || !rec || len <= 0 || !pp || !R || !pb || !L_out || !p || !tr || !pav) return fail(HHG_EINVAL, "hhg_query_from_a3m: bad argument");
  int32_t L = 0, N = 0, has_ss = 0;
  int rc = hhg_a3m_scan(rec, len, mp, &L, &N, &has_ss);
  if (rc != HHG_OK) return rc;
  if (L < 1 || L > L_cap) return fail(HHG_EINVAL, "hhg_query_from_a3m: query length %d exceeds the caller's capacity %d", L, L_cap);
  CK(cudaSetDevice(ctx->device));
  DevBuf<float> d_tr;
  CK(d_tr.alloc((size_t)(L + 1) * 7));
  hhg_db* db = nullptr;
  const int64_t zero = 0;
  float nh = 0.f;
  rc = db_create_a3m_impl(ctx, 1, rec, &zero, &len, nullptr, mp, S, pb, pp, R, &db, d_tr.p, &nh);
  if (rc != HHG_OK) return rc;
  std::unique_ptr<hhg_db> holder(db);
  std::vector<ColRec> cols((size_t)L);
  CK(cudaMemcpyAsync(cols.data(), db->cols_raw.p, (size_t)L * sizeof(ColRec), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(tr, d_tr.p, (size_t)(L + 1) * 28, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(pav, db->pav.p, 80, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int i = 1; i <= L; ++i) {
    memcpy(p + (size_t)i * 20, cols[i - 1].p, 80);
    if (ss) ss[i] = (uint8_t)cols[i - 1].ss;
  }
  memcpy(p, pav, 80);                               // CalculateAminoAcidBackground: p[0] = p[L+1] = pav (:1866)
  memcpy(p + (size_t)(L + 1) * 20, pav, 80);
  if (ss) ss[0] = ss[L + 1] = 0;
  if (neff) *neff = nh;
  *L_out = L;
  return HHG_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Context-specific pseudocounts of the query (hhg_crf.cuh)
}  // extern "C"
struct hhg_crf {
  int device = 0;
  hhg::CrfHost host;
  DevBuf<double> d_w, d_bias;
};
extern "C" {

int hhg_crf_create(hhg_ctx* ctx, const char* text, int64_t len, hhg_crf** out) {
  if (!ctx || !text || len <= 0 || !out) return fail(HHG_EINVAL, "hhg_crf_create: bad argument");
  std::unique_ptr<hhg_crf> c(new hhg_crf());
  const std::string msg = crf_parse(text, len, &c->host);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_crf_create: %s", msg.c_str());
  CK(cudaSetDevice(ctx->device));
  c->device = ctx->device;
  CK(c->d_w.alloc(c->host.w.size())); CK(c->d_bias.alloc(c->host.bias.size()));
  CK(cudaMemcpyAsync(c->d_w.p, c->host.w.data(), c->host.w.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(c->d_bias.p, c->host.bias.data(), c->host.bias.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *out = c.release();
  return HHG_OK;
}

int hhg_crf_destroy(hhg_crf* crf) { delete crf; return HHG_OK; }

int hhg_crf_info(const hhg_crf* crf, int32_t* n_states, int32_t* window, double* pc /* [n_states*20] or NULL */) {
  if (!crf || !n_states || !window) return fail(HHG_EINVAL, "hhg_crf_info: bad argument");
  *n_states = crf->host.K; *window = crf->host.W;
  if (pc) memcpy(pc, crf->host.pc.data(), crf->host.pc.size() * 8);
  return HHG_OK;
}

// Host only: the per-column tail of hhg_query_context_pseudocounts on caller-supplied context scores
// (score[L*K], what k_crf_scores produces), for inspection and CPU-side tests.
int hhg_crf_tail_host(const hhg_crf* crf, int32_t L, double* score, const float* f, const float* neff_m, const hhg_admix* admix,
                      float* p) {
  if (!crf || L < 1 || !score || !f || !neff_m || !admix || !p) return fail(HHG_EINVAL, "hhg_crf_tail_host: bad argument");
  const int K = crf->host.K;
  for (int i = 0; i < L; ++i) {
    double cnt[20];
    for (int a = 0; a < 20; ++a) cnt[a] = f[(size_t)(i + 1) * 20 + a] * neff_m[i + 1];
    crf_column_tail(K, score + (size_t)i * K, crf->host.pc.data(), cnt, (double)neff_m[i + 1], admix->kind, admix->pca, admix->pcb,
                    admix->pcc, p + (size_t)(i + 1) * 20);
  }
  return HHG_OK;
}

// Host only: parse without a device (no upload); for CPU-side tests of the parser and the tail.
int hhg_crf_parse_host(const char* text, int64_t len, hhg_crf** out) {
  if (!text || len <= 0 || !out) return fail(HHG_EINVAL, "hhg_crf_parse_host: bad argument");
  std::unique_ptr<hhg_crf> c(new hhg_crf());
  const std::string msg = crf_parse(text, len, &c->host);
  if (!msg.empty()) return fail(HHG_EINVAL, "hhg_crf_parse_host: %s", msg.c_str());
  *out = c.release();
  return HHG_OK;
}

// Host only: weights of one state, w[window*20] (row-major window x amino acid) and its bias.
int hhg_crf_state(const hhg_crf* crf, int32_t k, double* w, double* bias) {
  if (!crf || k < 0 || k >= crf->host.K || !w || !bias) return fail(HHG_EINVAL, "hhg_crf_state: bad argument");
  for (int j = 0; j < crf->host.W; ++j)
    for (int a = 0; a < 20; ++a) w[j * 20 + a] = crf->host.w[((size_t)j * 20 + a) * crf->host.K + k];
  *bias = crf->host.bias[k];
  return HHG_OK;
}

int hhg_query_context_pseudocounts(hhg_ctx* ctx, const hhg_crf* crf, int32_t L, const float* f, const float* neff_m,
                                   float neff_hmm, const float* pb, const hhg_admix* admix, float* p, float* pav) {
  if (!ctx || !crf || L < 1 || !f || !neff_m || !admix || !p) return fail(HHG_EINVAL, "hhg_query_context_pseudocounts: bad argument");
  if (admix->kind < 0 || admix->kind > 2) return fail(HHG_EINVAL, "hhg_query_context_pseudocounts: admixture kind %d (0 constant, 1 CS-BLAST, 2 HHsearch)", admix->kind);
  if (pav && !pb) return fail(HHG_EINVAL, "hhg_query_context_pseudocounts: pav needs the background pb");
  CK(cudaSetDevice(ctx->device));
  const int K = crf->host.K, W = crf->host.W;
  // HMM::fillCountProfile (src/hhhmm.cpp:1843-1849): counts = f * Neff_M (float product), neff = Neff_M
  std::vector<double> counts((size_t)L * 20), neff(L);
  for (int i = 0; i < L; ++i) {
    neff[i] = neff_m[i + 1];
    for (int a = 0; a < 20; ++a) counts[(size_t)i * 20 + a] = f[(size_t)(i + 1) * 20 + a] * neff_m[i + 1];
  }
  struct CrfStage {
    DevBuf<double> counts, score;
    double* h_score = nullptr; size_t h_n = 0;
    ~CrfStage() { if (h_score) cudaFreeHost(h_score); }
  };
  if (!ctx->crf_cache) ctx->crf_cache = std::make_shared<CrfStage>();
  CrfStage& st = *std::static_pointer_cast<CrfStage>(ctx->crf_cache);
  const size_t ns = (size_t)L * K;
  CK(st.counts.ensure(counts.size())); CK(st.score.ensure(ns));
  if (st.h_n < ns) {
    if (st.h_score) cudaFreeHost(st.h_score);
    st.h_score = nullptr; st.h_n = 0;
    CK(cudaHostAlloc((void**)&st.h_score, ns * 8, cudaHostAllocDefault));
    st.h_n = ns;
  }
  CK(cudaMemcpyAsync(st.counts.p, counts.data(), counts.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  k_crf_scores<<<dim3((K + 255) / 256, L), 256, 0, ctx->stream>>>(L, K, W, crf->d_w.p, crf->d_bias.p, st.counts.p, st.score.p);
  ctx->launches++;
  CK(cudaGetLastError());
  double* score = st.h_score;
  CK(cudaMemcpyAsync(score, st.score.p, ns * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  auto work = [&](unsigned w) {
    for (int i = (int)w; i < L; i += (int)hw)
      crf_column_tail(K, score + (size_t)i * K, crf->host.pc.data(), counts.data() + (size_t)i * 20, neff[i],
                      admix->kind, admix->pca, admix->pcb, admix->pcc, p + (size_t)(i + 1) * 20);
  };
  std::vector<std::thread> pool;
  for (unsigned w = 1; w < hw; ++w) pool.emplace_back(work, w);
  work(0);
  for (auto& th : pool) th.join();
  if (pav) {                               // HMM::CalculateAminoAcidBackground (src/hhhmm.cpp:1854-1868)
    float pv[20];
    for (int a = 0; a < 20; ++a) pv[a] = pb[a] * 100.0f / neff_hmm;
    for (int i = 1; i <= L; ++i) for (int a = 0; a < 20; ++a) pv[a] += p[(size_t)i * 20 + a];
    float sum = 0.0f;
    for (int a = 0; a < 20; ++a) sum += pv[a];
    if (sum != 0.0f) { const float fac = 1.0 / sum; for (int a = 0; a < 20; ++a) pv[a] *= fac; }
    memcpy(pav, pv, 80);
    memcpy(p, pv, 80); memcpy(p + (size_t)(L + 1) * 20, pv, 80);
  }
  return HHG_OK;
}

// The resident binary format: column records before the null model + pav.  read_* copy it out (to be stored
// next to the ffindex files), hhg_db_create_packed loads it back without parsing anything.
int hhg_db_read_cols(hhg_ctx* ctx, const hhg_db* db, int which, int64_t first, int64_t count, void* out) {
  if (!ctx || !db || !out || first < 0 || count < 0 || first + count > db->total_cols)
    return fail(HHG_EINVAL, "hhg_db_read_cols: bad argument");
  if (which != 0 && which != 1) return fail(HHG_EINVAL, "hhg_db_read_cols: which must be 0 (raw) or 1 (prepared)");
  if (which == 0 && !db->raw) return fail(HHG_EINVAL, "hhg_db_read_cols: db holds no pre-null-model records");
  if (which == 1 && !db->prepared) return fail(HHG_EINVAL, "hhg_db_read_cols: call hhg_db_apply_null_model first");
  CK(cudaSetDevice(ctx->device));
  const ColRec* src = reinterpret_cast<const ColRec*>(which == 0 ? db->cols_raw.p : db->cols.p) + first;
  CK(cudaMemcpyAsync(out, src, (size_t)count * sizeof(ColRec), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

int hhg_db_read_pav(hhg_ctx* ctx, const hhg_db* db, float* out) {
  if (!ctx || !db || !out || !db->raw) return fail(HHG_EINVAL, "hhg_db_read_pav: bad argument / db not raw");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(out, db->pav.p, (size_t)db->n * 20 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

int hhg_db_create_packed(hhg_ctx* ctx, int n, const int32_t* L, const void* cols_raw, int has_ss,
                         const float* pav, hhg_db** out) {
  if (!ctx || !out || n <= 0 || !L || !cols_raw || !pav) return fail(HHG_EINVAL, "hhg_db_create_packed: bad argument");
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<hhg_db> holder(new hhg_db());
  hhg_db* db = holder.get();
  db->device = ctx->device;
  db->n = n;
  db->has_ss = has_ss != 0;
  db->L.assign(L, L + n);
  db->col_off.resize(n);
  long long tot = 0;
  for (int k = 0; k < n; ++k) {
    if (L[k] < 1 || L[k] > 32767) return fail(HHG_EINVAL, "target %d: length %d out of [1,32767]", k, L[k]);
    db->col_off[k] = tot;
    tot += L[k];
  }
  db->total_cols = tot;
  cudaError_t e;
  if ((e = db->cols.alloc((size_t)tot * 7)) != cudaSuccess || (e = db->cols_raw.alloc((size_t)tot * 7)) != cudaSuccess ||
      (e = db->dL.alloc(n)) != cudaSuccess || (e = db->dcol_off.alloc(n)) != cudaSuccess ||
      (e = db->pav.alloc((size_t)n * 20)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_db_create_packed: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->dL.p, db->L.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->dcol_off.p, db->col_off.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->cols_raw.p, cols_raw, (size_t)tot * sizeof(ColRec), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->cols.p, db->cols_raw.p, (size_t)tot * sizeof(ColRec), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->pav.p, pav, (size_t)n * 20 * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  db->raw = true;
  db->prepared = false;
  *out = holder.release();
  return HHG_OK;
}

int hhg_debug_fastlog2_table(hhg_ctx* ctx, float* lg2_out) {
  if (!ctx || !lg2_out) return fail(HHG_EINVAL, "bad argument");
  memcpy(lg2_out, ctx->h_lg2.data(), 1025 * 4);
  return HHG_OK;
}

int hhg_db_destroy(hhg_db* db) {
  if (db) { cudaSetDevice(db->device); delete db; }
  return HHG_OK;
}
int hhg_db_size(const hhg_db* db) { return db ? db->n : 0; }
long long hhg_db_columns(const hhg_db* db) { return db ? db->total_cols : 0; }

int hhg_db_lengths(const hhg_db* db, int32_t* out) {
  if (!db || !out) return fail(HHG_EINVAL, "hhg_db_lengths: bad argument");
  memcpy(out, db->L.data(), (size_t)db->n * sizeof(int32_t));
  return HHG_OK;
}

// --------------------------------------------------------------------------------------- query
static int query_set_impl(hhg_ctx* ctx, int nq, const int32_t* Lq, const float* const* p, const float* const* tr,
                          const uint8_t* const* ss, const float* q_pav, const float* S33, const hhg_params* par) {
  if (!ctx || nq < 1 || !Lq || !p || !tr || !par) return fail(HHG_EINVAL, "hhg_query_set: bad argument");
  bool all_ss = ss != nullptr;
  for (int q = 0; q < nq; ++q) {
    if (Lq[q] < 1 || Lq[q] > 32767 || !p[q] || !tr[q]) return fail(HHG_EINVAL, "hhg_query_set: bad query %d", q);
    if (ss && !ss[q]) all_ss = false;
  }
  if (par->use_ss && (!all_ss || !S33)) return fail(HHG_EINVAL, "hhg_query_set: use_ss needs ss and S33");
  CK(cudaSetDevice(ctx->device));
  ctx->par = *par;
  ctx->nq = nq;
  ctx->q_L.assign(Lq, Lq + nq);
  ctx->q_row0.resize(nq);
  long long rows = 0;
  for (int q = 0; q < nq; ++q) {
    ctx->q_row0[q] = (int)rows;
    rows += (Lq[q] + 47) / 48 * 48;     // each query zero padded to a multiple of every strip height (8, 12, 16)
  }
  if (rows > 0x7fffffffLL / 7) return fail(HHG_EINVAL, "hhg_query_set: query batch too large");
  ctx->Lq = Lq[0];
  CK(ctx->qrec.ensure((size_t)rows * 7));
  CK(cudaMemsetAsync(ctx->qrec.p, 0, (size_t)rows * 112, ctx->stream));
  // pack with the same kernel as the DB (one-profile shards)
  for (int q = 0; q < nq; ++q) {
    std::vector<long long> col_off(1, 0);
    const int32_t L1 = Lq[q];
    const int64_t zero = 0;
    int rc = pack_profiles(ctx, 1, &L1, &zero, &zero, &zero, p[q], tr[q], ss ? ss[q] : nullptr, col_off, L1,
                           ctx->qrec.p + (size_t)ctx->q_row0[q] * 7);
    if (rc != HHG_OK) return rc;
  }
  ctx->has_ss = all_ss;
  ctx->has_S33 = false;
  if (S33) {
    CK(ctx->S33.ensure(44 * 44));
    CK(cudaMemcpyAsync(ctx->S33.p, S33, 44 * 44 * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->has_S33 = true;
  }
  ctx->has_q_pav = q_pav != nullptr;
  if (q_pav) {
    ctx->h_q_pav.assign(q_pav, q_pav + (size_t)nq * 20);
    CK(ctx->d_q_pav.ensure((size_t)nq * 20));
    CK(cudaMemcpyAsync(ctx->d_q_pav.p, q_pav, (size_t)nq * 80, cudaMemcpyHostToDevice, ctx->stream));
  }
  ctx->query_serial++;
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

int hhg_query_set(hhg_ctx* ctx, int Lq, const float* p, const float* tr, const uint8_t* ss,
                  const float* S33, const hhg_params* par) {
  const int32_t L1 = Lq;
  return query_set_impl(ctx, 1, &L1, &p, &tr, ss ? &ss : nullptr, nullptr, S33, par);
}

int hhg_query_set_batch(hhg_ctx* ctx, int nq, const int32_t* Lq, const float* const* p, const float* const* tr,
                        const uint8_t* const* ss, const float* q_pav, const float* S33, const hhg_params* par) {
  return query_set_impl(ctx, nq, Lq, p, tr, ss, q_pav, S33, par);
}

// Switch the PRED_PRED secondary-structure term on/off for the following searches without re-sending the query
// (Viterbi::Align picks the *AndSS kernels per 8-target batch, src/hhviterbirunner.cpp:14-26).
int hhg_set_use_ss(hhg_ctx* ctx, int use_ss) {
  if (!ctx) return fail(HHG_EINVAL, "ctx is NULL");
  if (use_ss && (!ctx->has_ss || !ctx->has_S33)) return fail(HHG_EINVAL, "hhg_set_use_ss: the query was set without ss / S33");
  ctx->par.use_ss = use_ss ? 1 : 0;
  return HHG_OK;
}

// ---------------------------------------------------------------------------------------- plan
// Strip height of a plan.  Whole-shard scans have work items to spare and take R = 16 (least per-column overhead,
// 253 GCUPS).  A small request (the few thousand survivors of the prefilter) is latency bound: its longest job is one
// serial sweep over Lmax columns per strip, so halving the strip height halves that critical path and doubles the
// number of work items that can run side by side.
static int plan_strip_rows(const hhg_ctx* ctx, const int32_t* req_query, int n) {
  if (ctx->R) return ctx->R;
  long long items16 = 0;
  if (!req_query) items16 = (long long)((n + 31) / 32) * ((ctx->q_L[0] + 15) / 16);
  else {
    std::vector<long long> cnt(ctx->nq, 0);
    for (int k = 0; k < n; ++k) if (req_query[k] >= 0 && req_query[k] < ctx->nq) cnt[req_query[k]]++;
    for (int q = 0; q < ctx->nq; ++q) items16 += (cnt[q] + 31) / 32 * ((ctx->q_L[q] + 15) / 16);
  }
  return items16 >= 4LL * ctx->sm_count * 8 ? 16 : 8;
}

// (Re)build a plan in place; device buffers only ever grow, so a plan object that is reused across
// searches (hhg_viterbi_search keeps one per context) does not touch cudaMalloc in steady state.
// req_query[k] = index (into the context's query batch) of the query request k is aligned with; NULL = query 0.
// Jobs never mix queries: the requests of each query are length-sorted and cut into 32-target jobs separately.
static int plan_build(hhg_ctx* ctx, hhg_plan* pl, const hhg_db* db, int n, const int32_t* ids,
                      const int32_t* req_query = nullptr) {
  if (!ctx || !db || n <= 0) return fail(HHG_EINVAL, "hhg_plan_create: bad argument");
  if (ctx->nq <= 0) return fail(HHG_EINVAL, "hhg_plan_create: no query set");
  if (db->device != ctx->device) return fail(HHG_EINVAL, "db lives on device %d, ctx on %d", db->device, ctx->device);
  CK(cudaSetDevice(ctx->device));
  const int R = plan_strip_rows(ctx, req_query, n);
  // the common case of a repeated request (same shard, same target list, same query batch geometry, e.g. every
  // query of a series against the whole shard) reuses the plan: no host sort, no uploads
  if (pl->db == db && pl->db_serial == db->serial && pl->n == n && pl->R == R && pl->q_L == ctx->q_L &&
      pl->q_row0 == ctx->q_row0 && !pl->ids.empty() && pl->max_bt_bytes == ctx->max_bt_bytes) {
    bool same = true;
    if (ids) same = memcmp(ids, pl->ids.data(), (size_t)n * 4) == 0;
    else for (int k = 0; k < n && same; ++k) same = pl->ids[k] == k;
    if (same) {
      if (req_query) same = memcmp(req_query, pl->req_query.data(), (size_t)n * 4) == 0;
      else for (int k = 0; k < n && same; ++k) same = pl->req_query[k] == 0;
    }
    if (same) { pl->celloff = false; return HHG_OK; }
  }
  pl->db = db;
  pl->db_serial = db->serial;
  pl->device = db->device;
  pl->max_bt_bytes = ctx->max_bt_bytes;
  pl->cells = pl->padded_cells = pl->alg_bytes = 0;
  pl->waves.clear();
  pl->celloff = false;
  pl->n = n;
  pl->R = R;
  pl->q_L = ctx->q_L; pl->q_row0 = ctx->q_row0;
  pl->Lq = ctx->q_L[0];
  pl->ids.resize(n); pl->req_query.resize(n);
  for (int k = 0; k < n; ++k) {
    const int id = ids ? ids[k] : k;
    if (id < 0 || id >= db->n) return fail(HHG_EINVAL, "request %d: target id %d out of range", k, id);
    const int q = req_query ? req_query[k] : 0;
    if (q < 0 || q >= ctx->nq) return fail(HHG_EINVAL, "request %d: query index %d out of range (batch of %d)", k, q, ctx->nq);
    pl->ids[k] = id; pl->req_query[k] = q;
  }
  // sort requests by (query, target length descending) (the length sort is what ViterbiRunner does per chunk,
  // src/hhviterbirunner.cpp:117-119; here it also makes LPT scheduling of the work queue)
  pl->order.resize(n);
  std::iota(pl->order.begin(), pl->order.end(), 0);
  std::stable_sort(pl->order.begin(), pl->order.end(), [&](int a, int b) {
    if (pl->req_query[a] != pl->req_query[b]) return pl->req_query[a] < pl->req_query[b];
    return db->L[pl->ids[a]] > db->L[pl->ids[b]];
  });
  // jobs: runs of up to 32 consecutive sorted requests of the same query
  std::vector<int> job_first, job_cnt;
  for (int k = 0; k < n;) {
    const int q = pl->req_query[pl->order[k]];
    int e = k;
    while (e < n && e - k < 32 && pl->req_query[pl->order[e]] == q) ++e;
    job_first.push_back(k); job_cnt.push_back(e - k);
    k = e;
  }
  pl->njobs = (int)job_first.size();
  pl->req_job.resize(n); pl->req_lane.resize(n);
  pl->job_Lmax.resize(pl->njobs); pl->job_query.resize(pl->njobs); pl->job_nstrips.resize(pl->njobs);
  pl->job_Lq.resize(pl->njobs); pl->job_qrow0.resize(pl->njobs); pl->job_ss_off.resize(pl->njobs);
  pl->job_bt_off.resize(pl->njobs); pl->job_bnd_off.resize(pl->njobs); pl->job_co_off.resize(pl->njobs);
  pl->job_jc_off.resize(pl->njobs);
  pl->jc_version = 0;
  std::vector<int> job_target((size_t)pl->njobs * 32);
  std::vector<int> req_Lt(n), req_Lq(n);
  long long bnd = 0, co = 0, jc = 0, ss = 0;
  size_t wave_bt = 0, max_wave_words = 0;   // words in the current wave
  Wave w;
  for (int jb = 0; jb < pl->njobs; ++jb) {
    const int first = job_first[jb], cnt = job_cnt[jb];
    const int q = pl->req_query[pl->order[first]];
    const int Lmax = db->L[pl->ids[pl->order[first]]];
    const int ns = (ctx->q_L[q] + R - 1) / R;
    pl->job_Lmax[jb] = Lmax; pl->job_query[jb] = q; pl->job_nstrips[jb] = ns;
    pl->job_Lq[jb] = ctx->q_L[q]; pl->job_qrow0[jb] = ctx->q_row0[q];
    for (int l = 0; l < 32; ++l) {
      const int rq = pl->order[first + std::min(l, cnt - 1)];   // padded lanes repeat the last target
      job_target[(size_t)jb * 32 + l] = pl->ids[rq];
      if (l < cnt) { pl->req_job[rq] = jb; pl->req_lane[rq] = l; }
    }
    const size_t words = (size_t)(ns * R / 4) * (Lmax + 1) * 32;
    if (wave_bt > 0 && (wave_bt + words) * 4 > ctx->max_bt_bytes) {
      w.job_end = jb;
      pl->waves.push_back(w);
      max_wave_words = std::max(max_wave_words, wave_bt);
      w.job_begin = jb;
      wave_bt = 0;
    }
    pl->job_bt_off[jb] = (long long)wave_bt;
    wave_bt += words;
    pl->job_bnd_off[jb] = bnd;
    bnd += (long long)(Lmax + 1) * 32;
    pl->job_co_off[jb] = co;
    pl->job_jc_off[jb] = jc;
    pl->job_ss_off[jb] = ss;
    jc += (long long)Lmax * 224;
    co += (long long)ns * (Lmax + 1) * 32;
    ss += ns;
    pl->padded_cells += (double)ns * R * (double)Lmax * 32.0;
  }
  w.job_end = pl->njobs;
  pl->waves.push_back(w);
  max_wave_words = std::max(max_wave_words, wave_bt);
  pl->ss_total = ss;
  pl->co_total = co;
  // work items (job, strip) of every wave in dispatch order: groups of G consecutive jobs, strip-major inside a group
  // (strip s of all the group's jobs, then strip s+1, ...), so consecutive strips of a job are G items apart
  pl->items.clear();
  for (Wave& wv : pl->waves) {
    wv.item_begin = (long long)pl->items.size();
    for (int g0 = wv.job_begin; g0 < wv.job_end; g0 += ctx->group_jobs) {
      const int g1 = std::min(g0 + ctx->group_jobs, wv.job_end);
      int maxns = 0;
      for (int jb = g0; jb < g1; ++jb) maxns = std::max(maxns, pl->job_nstrips[jb]);
      for (int sidx = 0; sidx < maxns; ++sidx)
        for (int jb = g0; jb < g1; ++jb)
          if (sidx < pl->job_nstrips[jb]) pl->items.push_back(make_int2(jb - wv.job_begin, sidx));
    }
    wv.item_end = (long long)pl->items.size();
  }
  pl->path_off.resize(n);
  long long po = 0;
  double cols_sum = 0;
  for (int k = 0; k < n; ++k) {
    const int Lt = db->L[pl->ids[k]];
    const int Lqk = ctx->q_L[pl->req_query[k]];
    req_Lt[k] = Lt; req_Lq[k] = Lqk;
    pl->path_off[k] = po;
    po += Lqk + Lt + 2;
    pl->cells += (double)Lqk * Lt;
    cols_sum += Lt;
  }
  if (po > 0x7fffffffLL) return fail(HHG_EINVAL, "plan too large: %lld path bytes (> 2^31-1); split the request", po);
  pl->path_total = po;
  pl->jc_total = jc;
  pl->alg_bytes = cols_sum * 112.0 + pl->cells * 1.0 + (double)sizeof(HitRec) * n;

  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  A(pl->d_job_target.ensure(job_target.size())); A(pl->d_job_Lmax.ensure(pl->njobs));
  A(pl->d_job_bt_off.ensure(pl->njobs)); A(pl->d_job_bnd_off.ensure(pl->njobs)); A(pl->d_job_co_off.ensure(pl->njobs));
  A(pl->d_job_jc_off.ensure(pl->njobs)); A(pl->d_jcols.ensure((size_t)jc));
  A(pl->d_job_query.ensure(pl->njobs)); A(pl->d_job_nstrips.ensure(pl->njobs)); A(pl->d_job_Lq.ensure(pl->njobs));
  A(pl->d_job_qrow0.ensure(pl->njobs)); A(pl->d_job_ss_off.ensure(pl->njobs)); A(pl->d_items.ensure(pl->items.size()));
  A(pl->d_req_job.ensure(n)); A(pl->d_req_lane.ensure(n)); A(pl->d_req_Lt.ensure(n)); A(pl->d_req_Lq.ensure(n));
  A(pl->d_path_off.ensure(n));
  A(pl->d_req_target.ensure(n)); A(pl->d_S.ensure((size_t)po));
  A(pl->d_bt.ensure(max_wave_words));
  { BndSlot* before = pl->d_bnd.p; A(pl->d_bnd.ensure((size_t)bnd));
    // fresh slots must not carry a bit pattern that looks like a valid tag (epochs start at 1)
    if (e == cudaSuccess && pl->d_bnd.p != before) A(cudaMemsetAsync(pl->d_bnd.p, 0, pl->d_bnd.n * sizeof(BndSlot), ctx->stream)); }
  A(pl->d_strip_score.ensure((size_t)ss * 32));
  A(pl->d_strip_ij.ensure((size_t)ss * 32));
  A(pl->d_counter.ensure(pl->waves.size()));
  A(pl->d_hits.ensure(n));
  A(pl->d_paths.ensure((size_t)po));
  if (e != cudaSuccess) return fail(HHG_ENOMEM, "hhg_plan_create: %s", cudaGetErrorString(e));

  cudaStream_t st = ctx->stream;
  auto H2D = [&](void* d, const void* h, size_t bytes) { return cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st); };
  CK(H2D(pl->d_job_target.p, job_target.data(), job_target.size() * 4));
  CK(H2D(pl->d_job_Lmax.p, pl->job_Lmax.data(), (size_t)pl->njobs * 4));
  CK(H2D(pl->d_job_bt_off.p, pl->job_bt_off.data(), (size_t)pl->njobs * 8));
  CK(H2D(pl->d_job_bnd_off.p, pl->job_bnd_off.data(), (size_t)pl->njobs * 8));
  CK(H2D(pl->d_job_co_off.p, pl->job_co_off.data(), (size_t)pl->njobs * 8));
  CK(H2D(pl->d_job_jc_off.p, pl->job_jc_off.data(), (size_t)pl->njobs * 8));
  CK(H2D(pl->d_job_query.p, pl->job_query.data(), (size_t)pl->njobs * 4));
  CK(H2D(pl->d_job_nstrips.p, pl->job_nstrips.data(), (size_t)pl->njobs * 4));
  CK(H2D(pl->d_job_Lq.p, pl->job_Lq.data(), (size_t)pl->njobs * 4));
  CK(H2D(pl->d_job_qrow0.p, pl->job_qrow0.data(), (size_t)pl->njobs * 4));
  CK(H2D(pl->d_job_ss_off.p, pl->job_ss_off.data(), (size_t)pl->njobs * 8));
  CK(H2D(pl->d_items.p, pl->items.data(), pl->items.size() * sizeof(int2)));
  CK(H2D(pl->d_req_job.p, pl->req_job.data(), (size_t)n * 4));
  CK(H2D(pl->d_req_lane.p, pl->req_lane.data(), (size_t)n * 4));
  CK(H2D(pl->d_req_Lt.p, req_Lt.data(), (size_t)n * 4));
  CK(H2D(pl->d_req_Lq.p, req_Lq.data(), (size_t)n * 4));
  CK(H2D(pl->d_req_target.p, pl->ids.data(), (size_t)n * 4));
  CK(H2D(pl->d_path_off.p, pl->path_off.data(), (size_t)n * 8));
  CK(cudaStreamSynchronize(st));
  return HHG_OK;
}

int hhg_plan_create(hhg_ctx* ctx, const hhg_db* db, int n, const int32_t* ids, hhg_plan** out) {
  if (!out) return fail(HHG_EINVAL, "hhg_plan_create: out is NULL");
  std::unique_ptr<hhg_plan> pl(new hhg_plan());
  int rc = plan_build(ctx, pl.get(), db, n, ids);
  if (rc != HHG_OK) return rc;
  *out = pl.release();
  return HHG_OK;
}

int hhg_plan_destroy(hhg_plan* plan) {
  if (plan) { if (plan->db) cudaSetDevice(plan->device); delete plan; }
  return HHG_OK;
}
double hhg_plan_cells(const hhg_plan* plan) { return plan ? plan->cells : 0; }
double hhg_plan_padded_cells(const hhg_plan* plan) { return plan ? plan->padded_cells : 0; }
double hhg_plan_algorithmic_bytes(const hhg_plan* plan) { return plan ? plan->alg_bytes : 0; }

static int set_exclusions(hhg_ctx* ctx, hhg_plan* pl, const int64_t* excl_off, const int32_t* excl_i,
                          const int32_t* excl_j) {
  pl->celloff = false;
  pl->n_excl_steps = 0;
  const long long total = excl_off ? excl_off[pl->n] : 0;
  const bool regions = !ctx->ex_q_lo.empty() || !ctx->ex_t_lo.empty();
  if (total <= 0 && !regions) return HHG_OK;
  const size_t co_words = (size_t)pl->co_total;
  CK(pl->d_co.ensure(co_words));
  CK(cudaMemsetAsync(pl->d_co.p, 0, co_words * 4, ctx->stream));
  if (total > 0) {
    // validate like hhg_mac_realign does: k_celloff_raster indexes the mask with these values
    if (excl_off[0] != 0) return fail(HHG_EINVAL, "excl_off[0] must be 0");
    if (!excl_i || !excl_j) return fail(HHG_EINVAL, "excl_i / excl_j are NULL");
    std::vector<int> sreq((size_t)total);
    for (int k = 0; k < pl->n; ++k) {
      if (excl_off[k + 1] < excl_off[k]) return fail(HHG_EINVAL, "excl_off is not monotonic at request %d", k);
      const int Lt = pl->db->L[pl->ids[k]];
      for (long long s = excl_off[k]; s < excl_off[k + 1]; ++s) {
        const int Lqk = pl->q_L[pl->req_query[k]];
        if (excl_i[s] < 1 || excl_i[s] > Lqk || excl_j[s] < 1 || excl_j[s] > Lt)
          return fail(HHG_EINVAL, "excluded step %lld of request %d is (%d,%d), outside 1..%d x 1..%d", s - excl_off[k], k,
                      excl_i[s], excl_j[s], Lqk, Lt);
        sreq[(size_t)s] = k;
      }
    }
    CK(pl->d_step_req.ensure((size_t)total)); CK(pl->d_step_i.ensure((size_t)total)); CK(pl->d_step_j.ensure((size_t)total));
    CK(cudaMemcpyAsync(pl->d_step_req.p, sreq.data(), (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(pl->d_step_i.p, excl_i, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(pl->d_step_j.p, excl_j, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 128;
    k_celloff_raster<<<(unsigned)((total + threads - 1) / threads), threads, 0, ctx->stream>>>(
        (int)total, pl->d_step_req.p, pl->d_step_i.p, pl->d_step_j.p, pl->d_req_job.p, pl->d_req_lane.p,
        pl->d_req_Lt.p, pl->d_req_Lq.p, pl->d_job_Lmax.p, pl->d_job_co_off.p, pl->R, pl->d_co.p);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));   // sreq is a host temporary
  }
  if (regions) {
    const int nq = (int)ctx->ex_q_lo.size(), nt = (int)ctx->ex_t_lo.size();
    std::vector<int> h;
    h.insert(h.end(), ctx->ex_q_lo.begin(), ctx->ex_q_lo.end()); h.insert(h.end(), ctx->ex_q_hi.begin(), ctx->ex_q_hi.end());
    h.insert(h.end(), ctx->ex_t_lo.begin(), ctx->ex_t_lo.end()); h.insert(h.end(), ctx->ex_t_hi.begin(), ctx->ex_t_hi.end());
    CK(ctx->d_ex.ensure(h.size()));
    CK(cudaMemcpyAsync(ctx->d_ex.p, h.data(), h.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    const int* d = ctx->d_ex.p;
    k_celloff_regions<<<(unsigned)((co_words + 255) / 256), 256, 0, ctx->stream>>>(
        (long long)co_words, pl->njobs, pl->d_job_co_off.p, pl->d_job_Lmax.p, pl->d_job_nstrips.p, pl->R, nq, d, d + nq,
        nt, d + 2 * nq, d + 2 * nq + nt, pl->d_co.p);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
  }
  pl->celloff = true;
  pl->n_excl_steps = (int)total;
  return HHG_OK;
}

// -excl / -template_excl (par.exclstr / par.template_exclstr): ranges of query rows / template columns that are switched
// off in every following search of this context (ViterbiRunner::exclude_regions, src/hhviterbirunner.cpp:291-330);
// n = 0 clears.  Ranges are 1-based and inclusive like the option strings.
int hhg_set_excluded_regions(hhg_ctx* ctx, int nq, const int32_t* q_lo, const int32_t* q_hi, int nt, const int32_t* t_lo,
                             const int32_t* t_hi) {
  if (!ctx || nq < 0 || nt < 0 || (nq && (!q_lo || !q_hi)) || (nt && (!t_lo || !t_hi)))
    return fail(HHG_EINVAL, "hhg_set_excluded_regions: bad argument");
  ctx->ex_q_lo.assign(q_lo, q_lo + nq); ctx->ex_q_hi.assign(q_hi, q_hi + nq);
  ctx->ex_t_lo.assign(t_lo, t_lo + nt); ctx->ex_t_hi.assign(t_hi, t_hi + nt);
  return HHG_OK;
}

}  // extern "C"

template <int R>
static int launch_viterbi(hhg_ctx* ctx, const VitParams& P, bool local, bool ss, bool co, int items) {
  const size_t smem = (size_t)kWarpsPerCta * R * 112 + 64 + (ss ? 44 * 44 * 4 : 0);
  void (*kern)(const VitParams) = nullptr;
#define PICK(L_, S_, C_) kern = k_viterbi<R, L_, S_, C_>
  if (local) { if (ss) { if (co) PICK(true, true, true); else PICK(true, true, false); }
               else    { if (co) PICK(true, false, true); else PICK(true, false, false); } }
  else       { if (ss) { if (co) PICK(false, true, true); else PICK(false, true, false); }
               else    { if (co) PICK(false, false, true); else PICK(false, false, false); } }
#undef PICK
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kWarpsPerCta * 32, smem));
  if (per_sm < 1) return fail(HHG_ECUDA, "viterbi kernel does not fit on an SM");
  // persistent grid: every CTA must be resident (strip items wait on their predecessor strip)
  int grid = ctx->sm_count * per_sm;
  const int need = (items + kWarpsPerCta - 1) / kWarpsPerCta;
  if (grid > need) grid = need;
  kern<<<grid, kWarpsPerCta * 32, smem, ctx->stream>>>(P);
  ctx->launches++;
  CK(cudaGetLastError());
  return HHG_OK;
}

extern "C" {

static int plan_run_impl(hhg_ctx* ctx, hhg_plan* pl, bool timed) {
  if (!ctx || !pl) return fail(HHG_EINVAL, "hhg_plan_run: bad argument");
  if (pl->q_L != ctx->q_L || pl->q_row0 != ctx->q_row0) return fail(HHG_EINVAL, "plan was made for another query (batch) geometry");
  const hhg_db* db = pl->db;
  const bool fused = pl->nm_mode >= 0;     // null model factored in per job while the operand stream is built
  if (fused && (!db->raw || !ctx->has_q_pav)) return fail(HHG_EINVAL, "fused null model needs a raw shard and query pav");
  if (!fused && !db->prepared) return fail(HHG_EINVAL, "raw db: call hhg_db_apply_null_model for the current query first");
  if (ctx->par.use_ss && (!db->has_ss || !ctx->has_ss || !ctx->has_S33))
    return fail(HHG_EINVAL, "use_ss requested but query/db/S33 carry no ss information");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // slot tags of earlier runs never match (20-bit epoch in the tag) ... unless the epoch has wrapped since this plan's
  // slots were last cleared: then a slot left over from exactly 2^20 runs ago would look valid, so clear them once
  // per epoch window
  ctx->epoch = (ctx->epoch + 1) & 0xFFFFFu;
  if (ctx->epoch == 0) { ctx->epoch = 1; ctx->epoch_window++; }
  if (pl->bnd_epoch_window != ctx->epoch_window) {
    if (pl->d_bnd.p) CK(cudaMemsetAsync(pl->d_bnd.p, 0, pl->d_bnd.n * sizeof(BndSlot), st));
    pl->bnd_epoch_window = ctx->epoch_window;
  }
  CK(cudaMemsetAsync(pl->d_counter.p, 0, pl->waves.size() * 4, st));
  if (pl->jc_version != db->cols_version || pl->jc_nm_mode != pl->nm_mode ||
      (fused && pl->jc_query_serial != ctx->query_serial)) {
    // (re)build the job-interleaved operand stream: once per plan, again after every hhg_db_apply_null_model (the
    // prepared emissions changed) and, with the fused null model, for every new query batch
    int maxL = 0;
    for (int jb = 0; jb < pl->njobs; ++jb) maxL = std::max(maxL, pl->job_Lmax[jb]);
    dim3 grid((unsigned)pl->njobs, (unsigned)std::min(64, (maxL + 7) / 8), 1);
    k_interleave_cols<<<grid, 256, 0, st>>>(pl->njobs, pl->d_job_target.p, pl->d_job_Lmax.p, pl->d_job_jc_off.p,
                                            fused ? db->cols_raw.p : db->cols.p, db->dcol_off.p, db->dL.p, pl->d_jcols.p,
                                            pl->nm_mode, pl->d_job_query.p, ctx->d_q_pav.p, db->pav.p, ctx->d_pb.p);
    ctx->launches++;
    CK(cudaGetLastError());
    pl->jc_version = db->cols_version;
    pl->jc_nm_mode = pl->nm_mode;
    pl->jc_query_serial = ctx->query_serial;
  }
  for (size_t wi = 0; wi < pl->waves.size(); ++wi) {
    const Wave& w = pl->waves[wi];
    const int nj = w.job_end - w.job_begin;
    VitParams P{};
    P.qrec = ctx->qrec.p;
    P.job_Lq = pl->d_job_Lq.p + w.job_begin; P.job_nstrips = pl->d_job_nstrips.p + w.job_begin;
    P.job_qrow0 = pl->d_job_qrow0.p + w.job_begin; P.job_ss_off = pl->d_job_ss_off.p + w.job_begin;
    P.items = pl->d_items.p + w.item_begin; P.n_items = (int)(w.item_end - w.item_begin);
    P.Lt = db->dL.p;
    P.jcols = pl->d_jcols.p;
    P.job_jc_off = pl->d_job_jc_off.p + w.job_begin;
    P.njobs = nj;
    P.job_target = pl->d_job_target.p + (size_t)w.job_begin * 32;
    P.job_Lmax = pl->d_job_Lmax.p + w.job_begin;
    P.job_bt_off = pl->d_job_bt_off.p + w.job_begin;
    P.job_bnd_off = pl->d_job_bnd_off.p + w.job_begin;
    P.job_co_off = pl->d_job_co_off.p + w.job_begin;
    P.bt = pl->d_bt.p; P.bnd = pl->d_bnd.p;
    P.tag_base = ctx->epoch << 12;
    P.counter = pl->d_counter.p + wi;
    P.strip_score = pl->d_strip_score.p;     // job_ss_off is absolute
    P.strip_ij = pl->d_strip_ij.p;
    P.celloff = pl->celloff ? pl->d_co.p : nullptr;
    P.S33 = ctx->has_S33 ? ctx->S33.p : nullptr;
    P.egq = ctx->par.egq; P.egt = ctx->par.egt; P.shift = ctx->par.shift; P.ssw = ctx->par.ssw;
    P.one2 = 0x3F8000003F800000ull;
    P.zero = 0u;

    const int items = P.n_items;
    int rc;
    if (timed) CK(cudaEventRecord(ctx->ev[0], st));
    if (pl->R == 8) rc = launch_viterbi<8>(ctx, P, ctx->par.local != 0, ctx->par.use_ss != 0, pl->celloff, items);
    else if (pl->R == 12) rc = launch_viterbi<12>(ctx, P, ctx->par.local != 0, ctx->par.use_ss != 0, pl->celloff, items);
    else rc = launch_viterbi<16>(ctx, P, ctx->par.local != 0, ctx->par.use_ss != 0, pl->celloff, items);
    if (rc != HHG_OK) return rc;
    if (timed) CK(cudaEventRecord(ctx->ev[1], st));
    // backtrace of this wave's requests.  Requests are addressed through the sorted order: the
    // wave covers sorted positions [req_begin, req_end); req_job/req_lane are per original request.
    BtParams B{};
    B.n_req = pl->n;   // filtered by job range inside: simpler to launch per wave over all requests
    B.job_nstrips = pl->d_job_nstrips.p; B.job_ss_off = pl->d_job_ss_off.p; B.job_qrow0 = pl->d_job_qrow0.p;
    B.nm_mode = pl->nm_mode; B.job_query = pl->d_job_query.p; B.q_pav = ctx->d_q_pav.p; B.t_pav = db->pav.p;
    B.pb = ctx->d_pb.p;
    B.req_job = pl->d_req_job.p; B.req_lane = pl->d_req_lane.p;
    B.job_Lmax = pl->d_job_Lmax.p; B.job_bt_off = pl->d_job_bt_off.p;
    B.bt = pl->d_bt.p; B.strip_score = pl->d_strip_score.p; B.strip_ij = pl->d_strip_ij.p;
    B.path_off = pl->d_path_off.p; B.hits = pl->d_hits.p; B.paths = pl->d_paths.p;
    B.job_begin = w.job_begin; B.job_end = w.job_end;
    B.req_target = pl->d_req_target.p; B.qrec = ctx->qrec.p; B.cols = fused ? db->cols_raw.p : db->cols.p; B.col_off = db->dcol_off.p;
    B.lg2 = ctx->lg2.p; B.diff = ctx->diff.p; B.S33 = ctx->has_S33 ? ctx->S33.p : nullptr; B.S = pl->d_S.p;
    B.corr = ctx->par.corr; B.ssw = ctx->par.ssw; B.use_ss = ctx->par.use_ss; B.ss_score_mode = (ctx->par.ssm == 2);
    const int threads = 128;
    k_backtrace<<<(pl->n + threads - 1) / threads, threads, 0, st>>>(B);
    ctx->launches++;
    CK(cudaGetLastError());
    if (timed) {
      CK(cudaEventRecord(ctx->ev[2], st));
      CK(cudaEventSynchronize(ctx->ev[2]));
      float a = 0, b = 0;
      CK(cudaEventElapsedTime(&a, ctx->ev[0], ctx->ev[1]));
      CK(cudaEventElapsedTime(&b, ctx->ev[1], ctx->ev[2]));
      pl->ms_viterbi += a;
      pl->ms_backtrace += b;
    }
  }
  return HHG_OK;
}

int hhg_plan_run(hhg_ctx* ctx, hhg_plan* pl) { return plan_run_impl(ctx, pl, false); }

// Same as hhg_plan_run but brackets every forward-pass and backtrace launch with CUDA events on the
// context stream and returns their summed device times (ms).  Synchronises; used by bench.py for the
// per-kernel roofline figure.
int hhg_plan_run_timed(hhg_ctx* ctx, hhg_plan* pl, float* ms_viterbi, float* ms_backtrace) {
  if (!ctx || !pl) return fail(HHG_EINVAL, "hhg_plan_run_timed: bad argument");
  for (int k = 0; k < 3; ++k)
    if (!ctx->ev[k]) CK(cudaEventCreate(&ctx->ev[k]));
  pl->ms_viterbi = pl->ms_backtrace = 0;
  int rc = plan_run_impl(ctx, pl, true);
  if (rc != HHG_OK) return rc;
  if (ms_viterbi) *ms_viterbi = pl->ms_viterbi;
  if (ms_backtrace) *ms_backtrace = pl->ms_backtrace;
  return HHG_OK;
}

int hhg_plan_fetch(hhg_ctx* ctx, hhg_plan* pl, hhg_hit* hits, uint8_t* paths, size_t paths_cap) {
  if (!ctx || !pl || !hits) return fail(HHG_EINVAL, "hhg_plan_fetch: bad argument");
  static_assert(sizeof(hhg_hit) == sizeof(HitRec), "hhg_hit / HitRec layout");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(hits, pl->d_hits.p, (size_t)pl->n * sizeof(HitRec), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (paths) {
    // compact on the device: only nsteps bytes per request cross PCIe (capacity is Lq+Lt+2 each)
    pl->h_compact_off.resize(pl->n);
    long long tot = 0;
    for (int k = 0; k < pl->n; ++k) { pl->h_compact_off[k] = tot; tot += hits[k].nsteps; }
    if (paths_cap < (size_t)tot) return fail(HHG_EINVAL, "paths buffer too small: need %lld bytes", tot);
    CK(pl->d_compact_off.ensure(pl->n));
    CK(pl->d_paths_compact.ensure((size_t)std::max<long long>(tot, 1)));
    CK(cudaMemcpyAsync(pl->d_compact_off.p, pl->h_compact_off.data(), (size_t)pl->n * 8, cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 128;
    k_gather_paths<<<(pl->n + threads - 1) / threads, threads, 0, ctx->stream>>>(
        pl->n, pl->d_hits.p, pl->d_path_off.p, pl->d_compact_off.p, pl->d_paths.p, pl->d_paths_compact.p);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(paths, pl->d_paths_compact.p, (size_t)tot, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < pl->n; ++k) hits[k].path_off = (int32_t)pl->h_compact_off[k];
  }
  return HHG_OK;
}

void* hhg_plan_hits_devptr(hhg_plan* plan) { return plan ? (void*)plan->d_hits.p : nullptr; }
hhg_plan* hhg_ctx_last_plan(hhg_ctx* ctx) { return ctx ? ctx->scratch_plan : nullptr; }

int hhg_plan_debug_bt(hhg_ctx* ctx, hhg_plan* pl, int k, uint8_t* bt) {
  if (!ctx || !pl || !bt || k < 0 || k >= pl->n) return fail(HHG_EINVAL, "hhg_plan_debug_bt: bad argument");
  if (pl->waves.size() != 1) return fail(HHG_EINVAL, "debug_bt needs a single-wave plan");
  CK(cudaSetDevice(ctx->device));
  const int job = pl->req_job[k], lane = pl->req_lane[k];
  const int Lt = pl->db->L[pl->ids[k]];
  const int Lqk = pl->q_L[pl->req_query[k]];
  const int total = (Lqk + 1) * (Lt + 1);
  DevBuf<uint8_t> tmp;
  CK(tmp.alloc(total));
  k_debug_bt<<<(total + 255) / 256, 256, 0, ctx->stream>>>(pl->d_bt.p, pl->job_bt_off[job], lane,
                                                            pl->job_Lmax[job], Lqk, Lt, tmp.p);
  ctx->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(bt, tmp.p, total, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

int hhg_viterbi_search(hhg_ctx* ctx, const hhg_db* db, int n, const int32_t* ids, hhg_hit* hits,
                       uint8_t* paths, size_t paths_cap, const int64_t* excl_off,
                       const int32_t* excl_i, const int32_t* excl_j) {
  if (!ctx) return fail(HHG_EINVAL, "ctx is NULL");
  if (!ctx->scratch_plan) ctx->scratch_plan = new hhg_plan();
  hhg_plan* pl = ctx->scratch_plan;
  static const bool timing = getenv("HHG_TIMING") != nullptr;   // developer aid: host-side phase times on stderr
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto t0 = now();
  int rc = plan_build(ctx, pl, db, n, ids);
  if (rc != HHG_OK) return rc;
  pl->nm_mode = -1;
  auto t1 = now();
  rc = set_exclusions(ctx, pl, excl_off, excl_i, excl_j);
  if (rc == HHG_OK) rc = hhg_plan_run(ctx, pl);
  if (timing) cudaStreamSynchronize(ctx->stream);
  auto t2 = now();
  if (rc == HHG_OK) rc = hhg_plan_fetch(ctx, pl, hits, paths, paths_cap);
  if (timing) {
    auto ms = [](decltype(t0) a, decltype(t0) b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    fprintf(stderr, "[hhg] viterbi_search n=%d: plan %.3f ms, run (device) %.3f ms, fetch %.3f ms\n", n, ms(t0, t1), ms(t1, t2), ms(t2, now()));
  }
  return rc;
}


// Query-batch search (SURVEY 8f-4): nq queries set by hhg_query_set_batch, request k aligns query req_query[k] with
// target ids[k]; ONE plan, one forward launch per memory wave with the work items of all queries in it.
int hhg_viterbi_search_batch(hhg_ctx* ctx, const hhg_db* db, int n, const int32_t* req_query, const int32_t* ids,
                             int columnscore, const float* pb, hhg_hit* hits, uint8_t* paths, size_t paths_cap) {
  if (!ctx || !db || !req_query || !ids) return fail(HHG_EINVAL, "hhg_viterbi_search_batch: bad argument");
  if (!ctx->scratch_plan) ctx->scratch_plan = new hhg_plan();
  hhg_plan* pl = ctx->scratch_plan;
  int rc = plan_build(ctx, pl, db, n, ids, req_query);
  if (rc != HHG_OK) return rc;
  pl->nm_mode = -1;
  if (db->raw) {
    // every query needs its own null model: factor it in while the plan's operand stream is built
    if (columnscore < 0 || columnscore > 3) return fail(HHG_EINVAL, "hhg_viterbi_search_batch: columnscore %d", columnscore);
    if (!ctx->has_q_pav) return fail(HHG_EINVAL, "hhg_viterbi_search_batch: raw shard needs q_pav in hhg_query_set_batch");
    if (columnscore == 0 && !pb) return fail(HHG_EINVAL, "hhg_viterbi_search_batch: columnscore 0 needs pb");
    float h[20] = {0};
    if (pb) memcpy(h, pb, 80);
    CK(ctx->d_pb.ensure(20));
    CK(cudaMemcpyAsync(ctx->d_pb.p, h, 80, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    pl->nm_mode = columnscore;
  }
  rc = set_exclusions(ctx, pl, nullptr, nullptr, nullptr);     // excluded regions of the context, if any
  if (rc == HHG_OK) rc = hhg_plan_run(ctx, pl);
  if (rc == HHG_OK) rc = hhg_plan_fetch(ctx, pl, hits, paths, paths_cap);
  return rc;
}

}  // extern "C"

// ------------------------------------------------------------------------------ multi-GPU: NCCL behind the C-ABI
// NCCL is bound at run time (dlopen "libnccl.so.2"): a single-GPU user needs no NCCL at all, and inside a process
// that already loaded a copy (e.g. PyTorch's bundled one) the same copy is used.  Only the stable core entry
// points are needed; their prototypes are restated here (nccl.h: ncclGetUniqueId :146, ncclCommInitRank :160,
// ncclCommDestroy :181, ncclAllGather :425, ncclAllReduce, ncclGetErrorString).
namespace {
typedef struct ncclComm* nccl_comm_t;
typedef struct { char internal[128]; } nccl_uid_t;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(nccl_uid_t*) = nullptr;
  int (*CommInitRank)(nccl_comm_t*, int, nccl_uid_t, int) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
std::once_flag g_nccl_once;
const char* g_nccl_err = nullptr;

int nccl_load() {
  std::call_once(g_nccl_once, [] {
    const char* names[] = {getenv("HHG_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      if (!nm) continue;
      g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) { g_nccl_err = "libnccl.so.2 not found (set HHG_NCCL_LIB)"; return; }
#define SYM(f) *(void**)(&g_nccl.f) = dlsym(g_nccl.lib, "nccl" #f); if (!g_nccl.f) g_nccl_err = "NCCL symbol nccl" #f " missing"
    SYM(GetUniqueId); SYM(CommInitRank); SYM(CommDestroy); SYM(AllGather); SYM(AllReduce); SYM(GetErrorString);
#undef SYM
  });
  return g_nccl_err ? fail(HHG_ECUDA, "%s", g_nccl_err) : HHG_OK;
}
#define NCK(expr)                                                                                           \
  do {                                                                                                      \
    int r__ = (expr);                                                                                       \
    if (r__ != 0) return fail(HHG_ECUDA, "%s: NCCL error %d (%s)", #expr, r__, g_nccl.GetErrorString(r__)); \
  } while (0)
}  // namespace

struct hhg_comm {
  int rank = 0, world = 1, device = 0;
  nccl_comm_t comm = nullptr;
};

extern "C" {

int hhg_comm_unique_id(void* id128) {
  if (!id128) return fail(HHG_EINVAL, "hhg_comm_unique_id: id is NULL");
  int rc = nccl_load();
  if (rc != HHG_OK) return rc;
  nccl_uid_t id;
  NCK(g_nccl.GetUniqueId(&id));
  memcpy(id128, &id, sizeof id);
  return HHG_OK;
}

int hhg_comm_create(hhg_ctx* ctx, int rank, int world, const void* id128, hhg_comm** out) {
  if (!ctx || !out || world < 1 || rank < 0 || rank >= world || (world > 1 && !id128))
    return fail(HHG_EINVAL, "hhg_comm_create: bad argument");
  std::unique_ptr<hhg_comm> c(new hhg_comm());
  c->rank = rank; c->world = world; c->device = ctx->device;
  if (world > 1) {
    int rc = nccl_load();
    if (rc != HHG_OK) return rc;
    CK(cudaSetDevice(ctx->device));
    nccl_uid_t id;
    memcpy(&id, id128, sizeof id);
    NCK(g_nccl.CommInitRank(&c->comm, world, id, rank));
  }
  *out = c.release();
  return HHG_OK;
}

int hhg_comm_destroy(hhg_comm* c) {
  if (!c) return HHG_OK;
  if (c->comm) { cudaSetDevice(c->device); g_nccl.CommDestroy(c->comm); }
  delete c;
  return HHG_OK;
}

int hhg_comm_rank(const hhg_comm* c) { return c ? c->rank : 0; }
int hhg_comm_world(const hhg_comm* c) { return c ? c->world : 1; }

// Top-K of the last run of `plan`, merged over all ranks of `comm` (NULL / world 1: this GPU only).
static int plan_topk_impl(hhg_ctx* ctx, hhg_plan* pl, hhg_comm* comm, int K, int by_hit_score, const float* user_key,
                          int32_t id_base, const int32_t* global_ids, hhg_topk_rec* out, int* n_out) {
  static_assert(sizeof(hhg_topk_rec) == sizeof(TopkRec), "hhg_topk_rec / TopkRec layout");
  if (!ctx || !pl || K < 1 || !out || !n_out) return fail(HHG_EINVAL, "hhg_plan_topk: bad argument");
  if (comm && comm->world > 1 && comm->device != ctx->device) return fail(HHG_EINVAL, "hhg_plan_topk: comm lives on another device");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int n = pl->n;
  const int world = comm ? comm->world : 1, rank = comm ? comm->rank : 0;
  const int kl = std::min(K, n);
  CK(pl->d_keys.ensure((size_t)n)); CK(pl->d_topk_state.ensure(1));
  CK(pl->d_topk_local.ensure((size_t)K)); CK(pl->d_topk_all.ensure((size_t)K * world));
  if (global_ids) {
    CK(pl->d_gids.ensure((size_t)n));
    CK(cudaMemcpyAsync(pl->d_gids.p, global_ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  }
  if (user_key) {
    CK(pl->d_user_key.ensure((size_t)n));
    CK(cudaMemcpyAsync(pl->d_user_key.p, user_key, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  }
  TopkState init{};
  init.krem = (unsigned)kl;
  CK(cudaMemcpyAsync(pl->d_topk_state.p, &init, sizeof init, cudaMemcpyHostToDevice, st));
  const int threads = 256, blocks = (n + threads - 1) / threads;
  k_topk_keys<<<blocks, threads, 0, st>>>(n, pl->d_hits.p, by_hit_score, id_base, global_ids ? pl->d_gids.p : nullptr,
                                            user_key ? pl->d_user_key.p : nullptr, pl->d_keys.p);
  const int hblocks = std::min(blocks, ctx->sm_count * 4);
  for (int p = 7; p >= 0; --p) {
    k_topk_hist<<<hblocks, threads, 0, st>>>(n, pl->d_keys.p, p, pl->d_topk_state.p);
    k_topk_scan<<<1, 256, 0, st>>>(pl->d_topk_state.p);
  }
  k_topk_emit<<<blocks, threads, 0, st>>>(n, pl->d_keys.p, pl->d_hits.p, rank, pl->d_topk_state.p, pl->d_topk_local.p, K);
  ctx->launches += 18;
  if (kl < K) { k_topk_pad<<<(K - kl + 255) / 256, 256, 0, st>>>(pl->d_topk_local.p, kl, K); ctx->launches++; }
  CK(cudaGetLastError());
  const TopkRec* src = pl->d_topk_local.p;
  if (world > 1) {
    NCK(g_nccl.AllGather(pl->d_topk_local.p, pl->d_topk_all.p, (size_t)K * sizeof(TopkRec), /*ncclChar*/ 0, comm->comm, st));
    src = pl->d_topk_all.p;
  }
  std::vector<TopkRec> all((size_t)K * world);
  CK(cudaMemcpyAsync(all.data(), src, all.size() * sizeof(TopkRec), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  // merge: keys are unique and totally ordered (score descending, global id ascending)
  all.erase(std::remove_if(all.begin(), all.end(), [](const TopkRec& r) { return r.target < 0; }), all.end());
  std::sort(all.begin(), all.end(), [](const TopkRec& a, const TopkRec& b) { return a.key < b.key; });
  const int m = (int)std::min<size_t>(all.size(), (size_t)K);
  memcpy(out, all.data(), (size_t)m * sizeof(TopkRec));
  *n_out = m;
  return HHG_OK;
}

int hhg_plan_topk(hhg_ctx* ctx, hhg_plan* pl, hhg_comm* comm, int K, int by_hit_score, int32_t id_base,
                  const int32_t* global_ids, hhg_topk_rec* out, int* n_out) {
  return plan_topk_impl(ctx, pl, comm, K, by_hit_score, nullptr, id_base, global_ids, out, n_out);
}

int hhg_plan_topk_by_key(hhg_ctx* ctx, hhg_plan* pl, hhg_comm* comm, int K, const float* key, int32_t id_base,
                         const int32_t* global_ids, hhg_topk_rec* out, int* n_out) {
  if (!key) return fail(HHG_EINVAL, "hhg_plan_topk_by_key: key is NULL");
  return plan_topk_impl(ctx, pl, comm, K, 0, key, id_base, global_ids, out, n_out);
}

// State strings of the merged list: out[r*width .. ] = path of recs[r] (nsteps bytes, zero padded), on every rank.
int hhg_plan_topk_paths(hhg_ctx* ctx, hhg_plan* pl, hhg_comm* comm, int n_rec, const hhg_topk_rec* recs, int width,
                        uint8_t* out) {
  if (!ctx || !pl || n_rec < 0 || !recs || width < 1 || !out) return fail(HHG_EINVAL, "hhg_plan_topk_paths: bad argument");
  if (n_rec == 0) return HHG_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int world = comm ? comm->world : 1, rank = comm ? comm->rank : 0;
  CK(pl->d_topk_all.ensure((size_t)n_rec));
  CK(pl->d_topk_paths.ensure((size_t)n_rec * width));
  CK(cudaMemcpyAsync(pl->d_topk_all.p, recs, (size_t)n_rec * sizeof(TopkRec), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(pl->d_topk_paths.p, 0, (size_t)n_rec * width, st));
  k_topk_paths<<<n_rec, 128, 0, st>>>(n_rec, pl->d_topk_all.p, rank, pl->d_paths.p, width, pl->d_topk_paths.p);
  ctx->launches++;
  CK(cudaGetLastError());
  if (world > 1)
    NCK(g_nccl.AllReduce(pl->d_topk_paths.p, pl->d_topk_paths.p, (size_t)n_rec * width, /*ncclUint8*/ 1, /*ncclSum*/ 0, comm->comm, st));
  CK(cudaMemcpyAsync(out, pl->d_topk_paths.p, (size_t)n_rec * width, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return HHG_OK;
}

}  // extern "C"

extern "C" {

// ------------------------------------------------------------------------------------ MAC realignment
// HMM::Log2LinTransitionProbs(1.0) (src/hhhmm.cpp:2305-2313) for host arrays: tr = pow(2.0f, 1.0f * tr), which with
// float arguments is the C library's powf.  Host only.
int hhg_log2lin(int64_t n, const float* in, float* out) {
  if (n < 0 || !in || !out) return fail(HHG_EINVAL, "hhg_log2lin: bad argument");
  for (int64_t k = 0; k < n; ++k) out[k] = ::powf(2.0f, 1.0f * in[k]);
  return HHG_OK;
}

int hhg_mac_query_set(hhg_ctx* ctx, int Lq, const float* q_p, const float* q_tr_lin) {
  if (!ctx || Lq < 1 || Lq > 32767 || !q_p || !q_tr_lin) return fail(HHG_EINVAL, "hhg_mac_query_set: bad argument");
  CK(cudaSetDevice(ctx->device));
  std::vector<float> tr(q_tr_lin, q_tr_lin + (size_t)(Lq + 1) * 7);
  // PosteriorDecoderRunner::initializeQueryHMMTransitions, src/hhposteriordecoderrunner.cpp:145-155
  // (enum order M2M,M2I,M2D,I2M,I2I,D2M,D2D)
  tr[1] = tr[2] = tr[3] = tr[4] = tr[5] = tr[6] = 0.0f;
  float* e = tr.data() + (size_t)Lq * 7;
  e[0] = 1.0f; e[1] = e[2] = e[3] = e[4] = 0.0f; e[5] = 1.0f; e[6] = 0.0f;
  CK(ctx->mac_qp.ensure((size_t)(Lq + 2) * 20)); CK(ctx->mac_qtr.ensure(tr.size()));
  CK(cudaMemcpyAsync(ctx->mac_qp.p, q_p, (size_t)(Lq + 2) * 80, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->mac_qtr.p, tr.data(), tr.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->mac_Lq = Lq;
  return HHG_OK;
}

int hhg_mac_realign(hhg_ctx* ctx, const hhg_db* db, int n, const int32_t* target, const int32_t* vit,
                    const int64_t* vit_off, const int32_t* vit_i, const int32_t* vit_j, const int64_t* excl_off,
                    const int32_t* excl_i, const int32_t* excl_j, const hhg_mac_params* par, hhg_mac_hit* hits,
                    int32_t* out_i, int32_t* out_j, uint8_t* out_states, float* out_post, size_t path_cap) {
  if (!ctx || !db || n <= 0 || !target || !vit || !vit_off || !vit_i || !vit_j || !par || !hits || !out_i || !out_j ||
      !out_states || !out_post)
    return fail(HHG_EINVAL, "hhg_mac_realign: bad argument");
  if (ctx->mac_Lq <= 0) return fail(HHG_EINVAL, "hhg_mac_realign: call hhg_mac_query_set first");
  if (!db->prepared) return fail(HHG_EINVAL, "hhg_mac_realign: shard has no null model applied");
  if (excl_off && (!excl_i || !excl_j)) return fail(HHG_EINVAL, "hhg_mac_realign: excl_off without excl_i/excl_j");
  CK(cudaSetDevice(ctx->device));
  const bool timing = getenv("HHG_MAC_TIMING") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [](std::chrono::steady_clock::time_point a) {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
  };
  const auto t_begin = now();
  double t_prep = 0, t_lin = 0, t_kern = 0;
  const int Lq = ctx->mac_Lq;
  static_assert(sizeof(MacHitOut) == sizeof(hhg_mac_hit), "hhg_mac_hit layout");
  std::vector<long long> rec0(n), tr_off(n), cell_off(n), row_off(n), path_off(n);
  std::vector<int> Lt(n);
  long long ntr = 0, ncell = 0, nrow = 0, npath = 0;
  for (int r = 0; r < n; ++r) {
    const int t = target[r];
    if (t < 0 || t >= db->n) return fail(HHG_EINVAL, "request %d: target id %d out of range", r, t);
    const int L = db->L[t];
    const int32_t* v = vit + (size_t)r * 5;
    const long long ns = vit_off[r + 1] - vit_off[r];
    if (v[4] != ns || ns < 0) return fail(HHG_EINVAL, "request %d: nsteps %d but %lld path entries", r, v[4], ns);
    if (v[0] < 1 || v[1] > Lq || v[0] > v[1] || v[2] < 1 || v[3] > L || v[2] > v[3])
      return fail(HHG_EINVAL, "request %d: Viterbi end points (%d-%d, %d-%d) outside 1..%d x 1..%d", r, v[0], v[1], v[2], v[3], Lq, L);
    for (long long s = vit_off[r]; s < vit_off[r + 1]; ++s)
      if (vit_i[s] < 1 || vit_i[s] > Lq || vit_j[s] < 1 || vit_j[s] > L)
        return fail(HHG_EINVAL, "request %d: Viterbi path leaves the matrix", r);
    if (excl_off)
      for (long long s = excl_off[r]; s < excl_off[r + 1]; ++s)
        if (excl_i[s] < 1 || excl_i[s] > Lq || excl_j[s] < 1 || excl_j[s] > L)
          return fail(HHG_EINVAL, "request %d: excluded alignment leaves the matrix", r);
    rec0[r] = db->col_off[t]; Lt[r] = L;
    tr_off[r] = ntr; ntr += (long long)(L + 1) * 7;
    cell_off[r] = ncell; ncell += (long long)(Lq + 1) * (L + 1);
    row_off[r] = nrow; nrow += 11LL * (L + 3) + (L + 3 + 7) / 8 + 1;   // + the cell-off row of the fallback path
    path_off[r] = npath; npath += (long long)Lq + L + 2;
  }
  if ((size_t)npath > path_cap) return fail(HHG_EINVAL, "hhg_mac_realign: path buffers hold %zu entries, %lld needed", path_cap, npath);
  const long long nvit = vit_off[n], nexcl = excl_off ? excl_off[n] : 0;
  // device staging: one int64 block {rec0, tr_off, cell_off, row_off, path_off, vit_off[n+1], excl_off[n+1]},
  // one int32 block {Lt, vit[5n], vit_i, vit_j, excl_i, excl_j}
  std::vector<long long> h64;
  h64.insert(h64.end(), rec0.begin(), rec0.end());
  h64.insert(h64.end(), tr_off.begin(), tr_off.end());
  h64.insert(h64.end(), cell_off.begin(), cell_off.end());
  h64.insert(h64.end(), row_off.begin(), row_off.end());
  h64.insert(h64.end(), path_off.begin(), path_off.end());
  for (int r = 0; r <= n; ++r) h64.push_back(vit_off[r] - vit_off[0]);
  for (int r = 0; r <= n; ++r) h64.push_back(excl_off ? excl_off[r] - excl_off[0] : 0);
  std::vector<int> h32;
  h32.insert(h32.end(), Lt.begin(), Lt.end());
  h32.insert(h32.end(), vit, vit + (size_t)n * 5);
  h32.insert(h32.end(), vit_i + vit_off[0], vit_i + vit_off[0] + nvit);
  h32.insert(h32.end(), vit_j + vit_off[0], vit_j + vit_off[0] + nvit);
  if (excl_off) {
    h32.insert(h32.end(), excl_i + excl_off[0], excl_i + excl_off[0] + (nexcl - excl_off[0]));
    h32.insert(h32.end(), excl_j + excl_off[0], excl_j + excl_off[0] + (nexcl - excl_off[0]));
  }
  const long long nex = excl_off ? nexcl - excl_off[0] : 0;
  CK(ctx->mac_i64.ensure(h64.size())); CK(ctx->mac_i32.ensure(h32.size()));
  CK(ctx->mac_ttr.ensure((size_t)ntr)); CK(ctx->mac_post.ensure((size_t)ncell)); CK(ctx->mac_off.ensure((size_t)ncell));
  CK(ctx->mac_bt.ensure((size_t)ncell)); CK(ctx->mac_rows.ensure((size_t)nrow)); CK(ctx->mac_scale.ensure((size_t)n * (Lq + 3)));
  CK(ctx->mac_out.ensure(n)); CK(ctx->mac_out_i.ensure((size_t)npath)); CK(ctx->mac_out_j.ensure((size_t)npath));
  CK(ctx->mac_out_states.ensure((size_t)npath)); CK(ctx->mac_out_post.ensure((size_t)npath));
  CK(cudaMemcpyAsync(ctx->mac_i64.p, h64.data(), h64.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->mac_i32.p, h32.data(), h32.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->mac_bt.p, 0, (size_t)ncell, ctx->stream));
  const long long* d64 = ctx->mac_i64.p;
  const int* d32 = ctx->mac_i32.p;
  MacArgs A{};
  A.n = n; A.Lq = Lq; A.local = par->local ? 1 : 0; A.mact = par->mact;
  { const char* e = getenv("HHG_MAC_BANDSCAN"); A.band_scan = (e && atoi(e) == 0) ? 0 : 1; }   // default on (2.5x); 0 = full-row scans
  A.Cshift = ::pow(2.0, par->shift);                       // src/hhforwardalgorithm.cpp:16
  A.q_p = ctx->mac_qp.p; A.q_tr = ctx->mac_qtr.p;
  A.cols = reinterpret_cast<const ColRec*>(db->cols.p);
  A.rec0 = d64; A.tr_off = d64 + n; A.cell_off = d64 + 2 * n; A.row_off = d64 + 3 * n; A.path_off = const_cast<long long*>(d64 + 4 * n);
  A.vit_off = d64 + 5 * n; A.excl_off = excl_off ? d64 + 5 * n + (n + 1) : nullptr;
  A.Lt = d32; A.vit = d32 + n; A.vit_i = d32 + 6 * n; A.vit_j = d32 + 6 * n + nvit;
  A.excl_i = d32 + 6 * n + 2 * nvit; A.excl_j = d32 + 6 * n + 2 * nvit + nex;
  A.t_tr = ctx->mac_ttr.p;
  A.post = ctx->mac_post.p; A.off = ctx->mac_off.p; A.bt = ctx->mac_bt.p; A.rows = ctx->mac_rows.p;
  A.scale = ctx->mac_scale.p; A.out = ctx->mac_out.p;
  A.out_i = ctx->mac_out_i.p; A.out_j = ctx->mac_out_j.p; A.out_states = ctx->mac_out_states.p; A.out_post = ctx->mac_out_post.p;
  t_prep = ms_since(t_begin);
  const auto t_lin0 = now();
  // template transitions in linear space: gather the log2 rows on the device, powf on the host (a few threads),
  // boundary rows as initializeForAlignment sets them, back to the device
  k_mac_gather_tr<<<dim3(8, n), 128, 0, ctx->stream>>>(n, A.cols, A.rec0, A.Lt, A.tr_off, ctx->mac_ttr.p);
  ctx->launches++;
  {
    std::vector<float> htr((size_t)ntr);
    CK(cudaMemcpyAsync(htr.data(), ctx->mac_ttr.p, (size_t)ntr * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    auto work = [&](unsigned w) {
      for (int r = (int)w; r < n; r += (int)hw) {
        float* tr = htr.data() + tr_off[r];
        const int L = Lt[r];
        for (int i = 1; i < L; ++i)
          for (int k = 0; k < 7; ++k) tr[(size_t)i * 7 + k] = ::powf(2.0f, 1.0f * tr[(size_t)i * 7 + k]);
        float* b = tr;                 // t.tr[0]: M2M = 1, everything else 0
        b[0] = 1.0f; b[1] = b[2] = b[3] = b[4] = b[5] = b[6] = 0.0f;
        float* e = tr + (size_t)L * 7; // t.tr[L]: M2M = D2M = 1
        e[0] = 1.0f; e[1] = e[2] = e[3] = e[4] = 0.0f; e[5] = 1.0f; e[6] = 0.0f;
      }
    };
    std::vector<std::thread> pool;
    for (unsigned w = 1; w < hw; ++w) pool.emplace_back(work, w);
    work(0);
    for (auto& th : pool) th.join();
    CK(cudaMemcpyAsync(ctx->mac_ttr.p, htr.data(), (size_t)ntr * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  t_lin = ms_since(t_lin0);
  const auto t_k0 = now();
  // -excl / -template_excl of the context apply to the realignment like they do to the Viterbi stage
  DevBuf<int> d_reg;
  if (!ctx->ex_q_lo.empty() || !ctx->ex_t_lo.empty()) {
    std::vector<int> hreg;
    hreg.insert(hreg.end(), ctx->ex_q_lo.begin(), ctx->ex_q_lo.end()); hreg.insert(hreg.end(), ctx->ex_q_hi.begin(), ctx->ex_q_hi.end());
    hreg.insert(hreg.end(), ctx->ex_t_lo.begin(), ctx->ex_t_lo.end()); hreg.insert(hreg.end(), ctx->ex_t_hi.begin(), ctx->ex_t_hi.end());
    CK(d_reg.alloc(hreg.size()));
    CK(cudaMemcpyAsync(d_reg.p, hreg.data(), hreg.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));            // hreg goes out of scope
    A.reg = d_reg.p; A.reg_nq = (int)ctx->ex_q_lo.size(); A.reg_nt = (int)ctx->ex_t_lo.size();
  }
  k_mac_band<<<n, 256, 0, ctx->stream>>>(A);
  {
    // working set in shared memory (117 bytes per template column).  Requests whose templates fit 64 KB (Lt <= ~555)
    // run 3 warps per SM on the main stream; longer ones get their own launch with a window of up to 200 KB on an
    // auxiliary stream so that they overlap the rest; beyond that the kernel falls back to the global scratch.
    const size_t kSmall = 64 * 1024, kLarge = 200 * 1024;
    std::vector<int> small_ids, large_ids;
    size_t small_need = 0, large_need = 0;
    for (int r = 0; r < n; ++r) {
      const size_t need = (size_t)117 * (Lt[r] + 3);
      if (need <= kSmall) { small_ids.push_back(r); small_need = std::max(small_need, need); }
      else { large_ids.push_back(r); large_need = std::max(large_need, need); }
    }
    CK(cudaFuncSetAttribute(k_mac_realign, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLarge));
    if (timing) { CK(ctx->mac_dbg.ensure((size_t)n * 12)); A.dbg = ctx->mac_dbg.p; }
    if (large_ids.empty()) {
      A.smem_rows = (int)small_need;
      k_mac_realign<<<n, 32, small_need, ctx->stream>>>(A);
      ctx->launches++;
    } else {
      std::vector<int> map(small_ids);
      map.insert(map.end(), large_ids.begin(), large_ids.end());
      CK(ctx->mac_map.ensure(map.size()));
      CK(cudaMemcpyAsync(ctx->mac_map.p, map.data(), map.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
      if (!ctx->aux_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->aux_ev[0], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->aux_ev[1], cudaEventDisableTiming));
      }
      CK(cudaEventRecord(ctx->aux_ev[0], ctx->stream));              // band + inputs ready
      CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_ev[0], 0));
      MacArgs AL = A;
      const size_t lsm = std::min(large_need, kLarge);
      AL.smem_rows = (int)lsm;
      AL.req_map = ctx->mac_map.p + small_ids.size();
      k_mac_realign<<<(unsigned)large_ids.size(), 32, lsm, ctx->aux_stream>>>(AL);
      CK(cudaEventRecord(ctx->aux_ev[1], ctx->aux_stream));
      if (!small_ids.empty()) {
        A.smem_rows = (int)small_need;
        A.req_map = ctx->mac_map.p;
        k_mac_realign<<<(unsigned)small_ids.size(), 32, small_need, ctx->stream>>>(A);
      }
      CK(cudaStreamWaitEvent(ctx->stream, ctx->aux_ev[1], 0));
      ctx->launches += small_ids.empty() ? 1 : 2;
    }
  }
  ctx->launches += 1;
  CK(cudaGetLastError());
  if (timing) { CK(cudaStreamSynchronize(ctx->stream)); t_kern = ms_since(t_k0); }
  const auto t_d0 = now();
  CK(cudaMemcpyAsync(hits, ctx->mac_out.p, (size_t)n * sizeof(MacHitOut), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out_i, ctx->mac_out_i.p, (size_t)npath * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out_j, ctx->mac_out_j.p, (size_t)npath * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out_states, ctx->mac_out_states.p, (size_t)npath, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out_post, ctx->mac_out_post.p, (size_t)npath * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (timing) {
    std::vector<long long> d((size_t)n * 12);
    CK(cudaMemcpy(d.data(), ctx->mac_dbg.p, d.size() * 8, cudaMemcpyDeviceToHost));
    int big = 0;
    for (int r = 1; r < n; ++r) if (Lt[r] > Lt[big]) big = r;
    for (int r : {0, big}) {
      fprintf(stderr, "  request %d (Lt=%d) Mcycles: fwdA %.2f fwdScan %.2f fwdEnd %.2f Pf %.2f bwdA %.2f bwdB %.2f bwdC %.2f macA %.2f macScan %.2f bt %.2f\n",
              r, Lt[r], d[r * 12 + 0] / 1e6, d[r * 12 + 1] / 1e6, d[r * 12 + 2] / 1e6, d[r * 12 + 3] / 1e6, d[r * 12 + 4] / 1e6,
              d[r * 12 + 5] / 1e6, d[r * 12 + 6] / 1e6, d[r * 12 + 7] / 1e6, d[r * 12 + 8] / 1e6, d[r * 12 + 9] / 1e6);
    }
  }
  if (timing)
    fprintf(stderr, "hhg_mac_realign: n=%d cells=%lld  prep+H2D %.2f ms, transitions (gather, powf, H2D) %.2f ms, "
            "kernels %.2f ms, D2H %.2f ms, total %.2f ms\n", n, ncell, t_prep, t_lin, t_kern, ms_since(t_d0), ms_since(t_begin));
  ctx->mac_cell_off = cell_off;
  ctx->mac_Lt = Lt;
  return HHG_OK;
}

int hhg_mac_debug_posterior(hhg_ctx* ctx, int request, float* out) {
  if (!ctx || !out || request < 0 || request >= (int)ctx->mac_cell_off.size())
    return fail(HHG_EINVAL, "hhg_mac_debug_posterior: bad argument");
  CK(cudaSetDevice(ctx->device));
  const size_t cells = (size_t)(ctx->mac_Lq + 1) * (ctx->mac_Lt[request] + 1);
  CK(cudaMemcpyAsync(out, ctx->mac_post.p + ctx->mac_cell_off[request], cells * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

// ------------------------------------------------------------------------------------ prefilter
int hhg_csdb_create(hhg_ctx* ctx, int n, const int32_t* L, const int64_t* off, const uint8_t* seq,
                    hhg_csdb** out) {
  if (!ctx || !out || n <= 0 || !L || !off || !seq) return fail(HHG_EINVAL, "hhg_csdb_create: bad argument");
  CK(cudaSetDevice(ctx->device));
  std::unique_ptr<hhg_csdb> holder(new hhg_csdb());
  hhg_csdb* db = holder.get();
  db->n = n;
  db->device = ctx->device;
  long long tot = 0;
  for (int k = 0; k < n; ++k) tot = std::max<long long>(tot, off[k] + L[k]);
  db->total = tot;
  cudaError_t e;
  if ((e = db->dL.alloc(n)) != cudaSuccess || (e = db->doff.alloc(n)) != cudaSuccess ||
      (e = db->seq.alloc((size_t)tot)) != cudaSuccess || (e = db->scores.alloc(n)) != cudaSuccess)
    return fail(HHG_ENOMEM, "hhg_csdb_create: %s", cudaGetErrorString(e));
  CK(cudaMemcpyAsync(db->dL.p, L, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->doff.p, off, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(db->seq.p, seq, (size_t)tot, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *out = holder.release();
  return HHG_OK;
}

int hhg_csdb_destroy(hhg_csdb* db) {
  if (db) { cudaSetDevice(db->device); delete db; }
  return HHG_OK;
}

}  // extern "C"

template <int WB>
static int launch_prefilter(hhg_ctx* ctx, const PfParams& P) {
  const size_t smem = (size_t)220 * WB * 32 * 4;
  auto kern = k_prefilter_ungapped<WB>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 512, smem));
  if (per_sm < 1) return fail(HHG_ECUDA, "prefilter kernel does not fit on an SM");
  kern<<<ctx->sm_count * per_sm, 512, smem, ctx->stream>>>(P);
  ctx->launches++;
  CK(cudaGetLastError());
  return HHG_OK;
}

// registers per lane of one query tile (64 positions per register): the smallest size that covers the query in one
// tile, else full 512-position tiles (225 KB of shared memory)
static int prefilter_wb(int Lq) {
  static const int kWB[] = {1, 2, 3, 4, 5, 6, 7, 8};
  for (int wb : kWB) if (Lq <= 64 * wb) return wb;
  return 8;
}

extern "C" {

int hhg_prefilter_ungapped_run(hhg_ctx* ctx, const hhg_csdb* db, int Lq, const uint8_t* prof_host,
                               int offset, int upload_profile) {
  if (!ctx || !db || Lq < 1 || offset < 0 || offset > 255) return fail(HHG_EINVAL, "hhg_prefilter_ungapped_run: bad argument");
  const int WB = prefilter_wb(Lq);
  const int tile_pos = 64 * WB;
  const int ntiles = (Lq + tile_pos - 1) / tile_pos;
  const size_t tile_words = (size_t)220 * WB * 32;
  CK(cudaSetDevice(ctx->device));
  if (upload_profile) {
    if (!prof_host) return fail(HHG_EINVAL, "profile is NULL");
    // repack [220][Lq] bytes into [tile][220][WB][32 lanes] words: lane l of a tile owns its positions
    // l*2WB .. +2WB-1; word w = (position l*2WB+w | position l*2WB+WB+w), each as the s16 value p - offset
    std::vector<uint32_t> packed(tile_words * ntiles);
    const uint32_t pad = (uint32_t)(uint16_t)(int16_t)(-offset);
    for (int t = 0; t < ntiles; ++t)
      for (int k = 0; k < 220; ++k)
        for (int w = 0; w < WB; ++w)
          for (int l = 0; l < 32; ++l) {
            const int plo = t * tile_pos + l * 2 * WB + w, phi = plo + WB;
            const uint32_t lo = plo < Lq ? (uint32_t)(uint16_t)(int16_t)((int)prof_host[(size_t)k * Lq + plo] - offset) : pad;
            const uint32_t hi = phi < Lq ? (uint32_t)(uint16_t)(int16_t)((int)prof_host[(size_t)k * Lq + phi] - offset) : pad;
            packed[(size_t)t * tile_words + ((size_t)k * WB + w) * 32 + l] = lo | (hi << 16);
          }
    CK(ctx->pf_prof.ensure(packed.size() * 4));
    CK(cudaMemcpyAsync(ctx->pf_prof.p, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  CK(ctx->pf_counter.ensure((size_t)ntiles));
  CK(cudaMemsetAsync(ctx->pf_counter.p, 0, 4 * (size_t)ntiles, ctx->stream));
  if (ntiles > 1) { CK(ctx->pf_edge[0].ensure((size_t)db->total)); CK(ctx->pf_edge[1].ensure((size_t)db->total)); }
  for (int t = 0; t < ntiles; ++t) {
    PfParams P{};
    P.n = db->n; P.L = db->dL.p; P.off = db->doff.p; P.seq = db->seq.p;
    P.prof32 = reinterpret_cast<const uint32_t*>(ctx->pf_prof.p) + (size_t)t * tile_words;
    P.offset = offset; P.tile = t; P.last_tile = (t == ntiles - 1);
    P.edge_in = ntiles > 1 ? ctx->pf_edge[(t + 1) & 1].p : nullptr;
    P.edge_out = ntiles > 1 ? ctx->pf_edge[t & 1].p : nullptr;
    P.scores = db->scores.p; P.counter = ctx->pf_counter.p + t;
    int rc;
    switch (WB) {
      case 1: rc = launch_prefilter<1>(ctx, P); break;
      case 2: rc = launch_prefilter<2>(ctx, P); break;
      case 3: rc = launch_prefilter<3>(ctx, P); break;
      case 4: rc = launch_prefilter<4>(ctx, P); break;
      case 5: rc = launch_prefilter<5>(ctx, P); break;
      case 6: rc = launch_prefilter<6>(ctx, P); break;
      case 7: rc = launch_prefilter<7>(ctx, P); break;
      default: rc = launch_prefilter<8>(ctx, P); break;
    }
    if (rc != HHG_OK) return rc;
  }
  return HHG_OK;
}

// Prefilter::Prefilter + init_prefilter (src/hhprefilter.cpp:28-47,314-335), the two set-up steps of the prefilter:
// (1) the column-state library: parse the text of cs219.lib (cs::ContextLibrary / ContextProfile::Read,
//     src/cs/context_profile-inl.h:81-141) and put it in linear space (cs::TransformToLin; the shipped file has
//     ISLOG F, i.e. probs = pow(2, -value/1000) in double, already linear) -> lib[k*20+a], a in the library's own
//     alphabet order A R N D C Q E G H I L K M F P S T W Y V (= the internal amino-acid order of HH-suite);
// (2) the sequences: one per ffindex entry of <db>_cs219, length = entry length - 1 (the NUL terminator).
int hhg_cs219_parse(const char* text, int64_t len, float* lib, int n_cap, int* n_states) {
  if (!text || len <= 0 || !lib || !n_states) return fail(HHG_EINVAL, "hhg_cs219_parse: bad argument");
  const char* p = text;
  const char* end = text + len;
  auto next_line = [&](const char*& b, const char*& e) {
    if (p >= end) return false;
    b = p;
    while (p < end && *p != '\n') ++p;
    e = p;
    if (p < end) ++p;
    return true;
  };
  int k = 0;
  bool is_log = false;
  const char *b, *e;
  while (next_line(b, e)) {
    if (e - b >= 5 && !strncmp(b, "ISLOG", 5)) { const char* q = b + 5; while (q < e && (*q == ' ' || *q == '\t')) ++q; is_log = (q < e && *q == 'T'); }
    if (e - b >= 5 && !strncmp(b, "PROBS", 5)) {
      if (!next_line(b, e)) break;                       // the row of the central (only) column: index + 20 values
      if (k >= n_cap) return fail(HHG_EINVAL, "hhg_cs219_parse: more than %d states", n_cap);
      const char* q = b;
      while (q < e && (*q == ' ' || *q == '\t')) ++q;
      while (q < e && *q >= '0' && *q <= '9') ++q;         // column index
      for (int a = 0; a < 20; ++a) {
        while (q < e && (*q == ' ' || *q == '\t')) ++q;
        if (q >= e) return fail(HHG_EINVAL, "hhg_cs219_parse: state %d has fewer than 20 values", k);
        double prob;
        if (*q == '*') { prob = 0.0; ++q; }
        else {
          long v = 0; bool neg = false;
          if (*q == '-') { neg = true; ++q; }
          if (q >= e || *q < '0' || *q > '9') return fail(HHG_EINVAL, "hhg_cs219_parse: state %d: not a number", k);
          while (q < e && *q >= '0' && *q <= '9') v = v * 10 + (*q++ - '0');
          if (neg) v = -v;
          prob = pow(2, static_cast<double>(-v) / 1000.0);      // ContextProfile::Read, kScale = 1000
          if (is_log) prob = exp(log(prob));                       // read as log, then TransformToLin
        }
        lib[(size_t)k * 20 + a] = (float)prob;
      }
      ++k;
    }
  }
  if (k == 0) return fail(HHG_EINVAL, "hhg_cs219_parse: no ContextProfile found");
  *n_states = k;
  return HHG_OK;
}

int hhg_csdb_create_ffindex(hhg_ctx* ctx, int n, const char* data, const int64_t* off, const int64_t* len, hhg_csdb** out) {
  if (!ctx || n <= 0 || !data || !off || !len || !out) return fail(HHG_EINVAL, "hhg_csdb_create_ffindex: bad argument");
  std::vector<int32_t> L(n);
  std::vector<int64_t> o(n);
  std::vector<uint8_t> seq;
  size_t tot = 0;
  for (int k = 0; k < n; ++k) {
    if (len[k] < 1 || off[k] < 0) return fail(HHG_EINVAL, "hhg_csdb_create_ffindex: entry %d has length %lld", k, (long long)len[k]);
    tot += (size_t)len[k] - 1;
  }
  seq.reserve(tot);
  for (int k = 0; k < n; ++k) {
    L[k] = (int32_t)(len[k] - 1);                        // length[n] = entry->length - 1, :328
    o[k] = (int64_t)seq.size();
    seq.insert(seq.end(), (const uint8_t*)data + off[k], (const uint8_t*)data + off[k] + L[k]);
  }
  return hhg_csdb_create(ctx, n, L.data(), o.data(), seq.data(), out);
}

// Host-side query profile of the prefilter (once per query; Prefilter::stripe_query_profile,
// src/hhprefilter.cpp:356-424) in the LINEAR layout prof[k*Lq+pos]: 219 column states + the ANY state.
// q_p is HMM::p of the (prefilter-pseudocount) query, i.e. float[(Lq+2)*20]; note the reference indexes
// the 1-based p array with a 0-based position (SURVEY App. D-4), reproduced here.  lib219: the 219x20
// linear column-state probabilities of cs219.lib (cs::TransformToLin).
static inline float flog2_host(float x) {       // flog2, src/util-inl.h:83-93 (double polynomial constants)
  if (x <= 0) return -128;
  uint32_t u; memcpy(&u, &x, 4);
  float e = (float)((int)((u & 0x7F800000u) >> 23) - 0x7f);
  u = (u & 0x007FFFFFu) | 0x3f800000u; memcpy(&x, &u, 4);
  x -= 1.0;
  x *= (1.441740 + x * (-0.7077702 + x * (0.4123442 + x * (-0.1903190 + x * 0.0440047))));
  return x + e;
}

int hhg_prefilter_build_profile(int Lq, const float* q_p, const float* q_pav, const float* lib219,
                                int score_offset, int bit_factor, uint8_t* prof) {
  if (Lq < 1 || !q_p || !q_pav || !lib219 || !prof) return fail(HHG_EINVAL, "hhg_prefilter_build_profile: bad argument");
  for (int k = 0; k < 219; ++k)
    for (int pos = 0; pos < Lq; ++pos) {
      float sum = 0;
      for (int a = 0; a < 20; ++a) sum += ((q_p[(size_t)pos * 20 + a] * lib219[k * 20 + a]) / q_pav[a]);
      float dummy = flog2_host(sum) * bit_factor + score_offset + 0.5;
      prof[(size_t)k * Lq + pos] = dummy > 255.0 ? 255 : (dummy < 0 ? 0 : (uint8_t)dummy);
    }
  for (int pos = 0; pos < Lq; ++pos) prof[(size_t)219 * Lq + pos] = (uint8_t)(score_offset - 1);
  return HHG_OK;
}

// Stage-1 length correction of Prefilter::prefilter_db (src/hhprefilter.cpp:477).
int hhg_prefilter_corrected_score(int raw, int Lq, int Lt, int bit_factor) {
  return raw - (int)(bit_factor * (flog2_host((float)Lq) + flog2_host((float)Lt)));
}

// Stage-2 E-value of Prefilter::prefilter_db (src/hhprefilter.cpp:529):
//   evalue = (double)num_dbs * LQ * length * fpow2(-score / bit_factor)   with INTEGER division (App. D-6)
// fpow2: src/util-inl.h:190-214.
static inline float fpow2_host(float x) {
  if (x >= FLT_MAX_EXP) return FLT_MAX;
  if (x <= FLT_MIN_EXP) return 0.0f;
  float tx = (x - 0.5f) + (3 << 22);
  uint32_t ut; memcpy(&ut, &tx, 4);
  int lx = (int)(ut - 0x4b400000u);
  float dx = x - (float)lx;
  x = 1.0f + dx * (0.693019f + dx * (0.241404f + dx * (0.0520749f + dx * 0.0134929f)));
  uint32_t ux; memcpy(&ux, &x, 4);
  ux += ((uint32_t)lx << 23);
  memcpy(&x, &ux, 4);
  return x;
}

double hhg_prefilter_evalue(int score, long long num_dbs, int Lq, int Lt, int bit_factor) {
  const double factor = (double)num_dbs * Lq;
  return factor * Lt * fpow2_host(-score / bit_factor);
}

// Batch forms of the two host-side formulas (1M-sequence shards: no per-element FFI calls).
int hhg_prefilter_corrected_scores(int n, const int32_t* raw, const int32_t* L, int Lq, int bit_factor,
                                   int32_t* out) {
  if (n < 0 || !raw || !L || !out) return fail(HHG_EINVAL, "hhg_prefilter_corrected_scores: bad argument");
  const float lq = flog2_host((float)Lq);
  for (int k = 0; k < n; ++k) out[k] = raw[k] - (int)(bit_factor * (lq + flog2_host((float)L[k])));
  return HHG_OK;
}

int hhg_prefilter_evalues(int n, const int32_t* score, const int32_t* L, long long num_dbs, int Lq,
                          int bit_factor, double* out) {
  if (n < 0 || !score || !L || !out) return fail(HHG_EINVAL, "hhg_prefilter_evalues: bad argument");
  for (int k = 0; k < n; ++k) out[k] = hhg_prefilter_evalue(score[k], num_dbs, Lq, L[k], bit_factor);
  return HHG_OK;
}

// Gapped stage 2 on the GPU for `n` selected sequences (ids == NULL: the first n of the shard).
// gap_open is the reference's gapOpen argument = prefilter_gap_open + prefilter_gap_extend (:456).
int hhg_prefilter_sw(hhg_ctx* ctx, const hhg_csdb* db, int n, const int32_t* ids, int Lq,
                     const uint8_t* prof, int gap_open, int gap_extend, int bias, int32_t* scores) {
  if (!ctx || !db || n < 1 || Lq < 1 || !prof || !scores) return fail(HHG_EINVAL, "hhg_prefilter_sw: bad argument");
  const int W = (Lq + 31) / 32;
  const size_t prof_bytes = (size_t)220 * W * 32;
  const size_t work_bytes = (size_t)8 * 3 * W * 32;             // H/H/E columns of the 8 warps of a CTA
  const bool prof_smem = prof_bytes + work_bytes <= 227 * 1024;   // else the striped profile is read through L1/L2
  const size_t smem = (prof_smem ? prof_bytes : 0) + work_bytes;
  if (smem > 227 * 1024) return fail(HHG_EINVAL, "prefilter sw: query length %d too long (working columns exceed shared memory)", Lq);
  CK(cudaSetDevice(ctx->device));
  for (int k = 0; ids && k < n; ++k)
    if (ids[k] < 0 || ids[k] >= db->n) return fail(HHG_EINVAL, "prefilter sw: id %d out of range", ids[k]);
  std::vector<uint8_t> striped(prof_bytes);
  for (int k = 0; k < 220; ++k)
    for (int j = 0; j < W; ++j)
      for (int l = 0; l < 32; ++l) {
        const int pos = l * W + j;
        striped[((size_t)k * W + j) * 32 + l] = pos < Lq ? prof[(size_t)k * Lq + pos] : (uint8_t)bias;
      }
  CK(ctx->sw_prof.ensure(prof_bytes)); CK(ctx->sw_scores.ensure(n)); CK(ctx->pf_counter.ensure(1));
  if (ids) CK(ctx->sw_ids.ensure(n));
  CK(cudaMemcpyAsync(ctx->sw_prof.p, striped.data(), prof_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (ids) CK(cudaMemcpyAsync(ctx->sw_ids.p, ids, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->pf_counter.p, 0, 4, ctx->stream));
  SwParams P{};
  P.n = n; P.ids = ids ? ctx->sw_ids.p : nullptr; P.L = db->dL.p; P.off = db->doff.p; P.seq = db->seq.p;
  P.prof = ctx->sw_prof.p; P.W = W; P.gap_open = gap_open; P.gap_extend = gap_extend; P.bias = bias;
  P.scores = ctx->sw_scores.p; P.counter = ctx->pf_counter.p;
  void (*swk)(const SwParams) = prof_smem ? k_prefilter_sw<true> : k_prefilter_sw<false>;
  CK(cudaFuncSetAttribute(swk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, swk, 256, smem));
  if (per_sm < 1) return fail(HHG_ECUDA, "prefilter sw kernel does not fit on an SM");
  const int grid = std::min(ctx->sm_count * per_sm, (n + 7) / 8);
  swk<<<grid, 256, smem, ctx->stream>>>(P);
  ctx->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(scores, ctx->sw_scores.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));   // `striped` is a host temporary
  return HHG_OK;
}

// Stage 1 of Prefilter::prefilter_db selected on the device (src/hhprefilter.cpp:477-506).  The raw ungapped
// scores of the last hhg_prefilter_ungapped_run on this shard are corrected and histogrammed in one pass, the
// cut is read off the histogram, survivors are compacted and only they travel to the host, where they are put
// in the reference's order (descending by (score, index): comparePair + reverse, :489-490).
int hhg_prefilter_select(hhg_ctx* ctx, const hhg_csdb* db, int Lq, int bit_factor, int smax_thresh,
                         int min_hits, int32_t* ids, int32_t* scores, int cap, int* n_out) {
  if (!ctx || !db || Lq < 1 || min_hits < 0 || !ids || !scores || cap < 0 || !n_out)
    return fail(HHG_EINVAL, "hhg_prefilter_select: bad argument");
  CK(cudaSetDevice(ctx->device));
  const int n = db->n;
  CK(ctx->pf_corr.ensure(n)); CK(ctx->pf_ids_a.ensure(n)); CK(ctx->pf_score_a.ensure(n)); CK(ctx->pf_ids_b.ensure(n));
  CK(ctx->pf_hist.ensure(kPfHistBins + 2));
  CK(cudaMemsetAsync(ctx->pf_hist.p, 0, (kPfHistBins + 2) * 4, ctx->stream));
  const int blocks = std::min((n + 255) / 256, ctx->sm_count * 8);
  k_pf_correct_hist<<<blocks, 256, 0, ctx->stream>>>(n, db->dL.p, db->scores.p, flog2_host((float)Lq), bit_factor,
                                                     ctx->pf_corr.p, ctx->pf_hist.p);
  ctx->launches++;
  std::vector<unsigned> hist(kPfHistBins);
  CK(cudaMemcpyAsync(hist.data(), ctx->pf_hist.p, kPfHistBins * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  // keep while count < min_hits or score > smax_thresh  ==  everything above the threshold, but at least the
  // min_hits best: cut = min(smax_thresh, score of the min_hits-th best); ties at the cut resolved by index
  long long n_gt = 0;
  auto bin_of = [](long long score) { return (int)std::min<long long>(std::max<long long>(score + kPfHistBias, 0), kPfHistBins - 1); };
  if (bin_of(smax_thresh) <= 0 || bin_of(smax_thresh) >= kPfHistBins - 1)
    return fail(HHG_EINVAL, "hhg_prefilter_select: smax_thresh %d outside the histogram range", smax_thresh);
  for (int b = bin_of(smax_thresh) + 1; b < kPfHistBins; ++b) n_gt += hist[b];
  int cut = smax_thresh, take_eq = 0;
  long long want_eq = 0;
  const long long need = std::min<long long>(min_hits, n);
  if (n_gt < need) {
    long long above = 0;
    int b = kPfHistBins - 1;
    for (; b >= 0; --b) {                         // highest score whose class completes the first `need` entries
      if (above + hist[b] >= need) break;
      above += hist[b];
    }
    if (b <= 0 || b >= kPfHistBins - 1)
      return fail(HHG_EINVAL, "hhg_prefilter_select: corrected scores leave the histogram range");
    cut = b - kPfHistBias; take_eq = 1; want_eq = need - above;
  }
  CK(cudaMemsetAsync(ctx->pf_hist.p + kPfHistBins, 0, 8, ctx->stream));
  k_pf_compact<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, ctx->pf_corr.p, cut, take_eq, ctx->pf_ids_a.p,
                                                         ctx->pf_score_a.p, ctx->pf_ids_b.p,
                                                         ctx->pf_hist.p + kPfHistBins);
  ctx->launches++;
  CK(cudaGetLastError());
  unsigned cnt[2] = {0, 0};
  CK(cudaMemcpyAsync(cnt, ctx->pf_hist.p + kPfHistBins, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<int32_t> a(cnt[0]), sa(cnt[0]), b(cnt[1]);
  if (cnt[0]) {
    CK(cudaMemcpyAsync(a.data(), ctx->pf_ids_a.p, (size_t)cnt[0] * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(sa.data(), ctx->pf_score_a.p, (size_t)cnt[0] * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (cnt[1]) CK(cudaMemcpyAsync(b.data(), ctx->pf_ids_b.p, (size_t)cnt[1] * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  std::sort(b.begin(), b.end(), std::greater<int32_t>());        // ties at the cut: larger index first
  if ((long long)b.size() > want_eq) b.resize((size_t)want_eq);
  const long long total = (long long)a.size() + (long long)b.size();
  *n_out = (int)total;
  if (total > cap) return fail(HHG_EINVAL, "hhg_prefilter_select: %lld survivors exceed the output capacity %d", total, cap);
  std::vector<std::pair<int32_t, int32_t>> v;                     // (score, index), descending
  v.reserve((size_t)total);
  for (size_t k = 0; k < a.size(); ++k) v.emplace_back(sa[k], a[k]);
  std::sort(v.begin(), v.end(), std::greater<std::pair<int32_t, int32_t>>());
  for (int32_t id : b) v.emplace_back(cut, id);                   // below all of list A, already index-descending
  for (size_t k = 0; k < v.size(); ++k) { ids[k] = v[k].second; scores[k] = v[k].first; }
  return HHG_OK;
}

int hhg_prefilter_fetch(hhg_ctx* ctx, const hhg_csdb* db, int32_t* scores) {
  if (!ctx || !db || !scores) return fail(HHG_EINVAL, "hhg_prefilter_fetch: bad argument");
  CK(cudaMemcpyAsync(scores, db->scores.p, (size_t)db->n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HHG_OK;
}

int hhg_prefilter_ungapped(hhg_ctx* ctx, const hhg_csdb* db, int Lq, const uint8_t* prof, int offset,
                           int32_t* scores) {
  int rc = hhg_prefilter_ungapped_run(ctx, db, Lq, prof, offset, 1);
  if (rc != HHG_OK) return rc;
  return hhg_prefilter_fetch(ctx, db, scores);
}

}  // extern "C"
