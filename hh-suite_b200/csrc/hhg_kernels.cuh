// hh-suite_b200/csrc/hhg_kernels.cuh -- sm_100a kernels of the HH-suite hot path.
//
// Viterbi HMM-HMM forward pass (replaces Viterbi::AlignWith[Out]CellOff[AndSS],
// /root/reference/src/hhviterbialgorithm.cpp:29-497) and the byte backtrace
// (Viterbi::Backtrace, src/hhviterbi.cpp:83-160).
//
// Mapping (B200-first, not the reference's 8-lane AVX2 row sweep):
//   * one LANE = one target; one WARP-JOB = 32 length-sorted targets; the job's DP matrix is cut
//     into STRIPS of R query rows.  A work item is (job, strip); persistent warps pull items from
//     an atomic queue in (job, strip) order, so consecutive strips of a job run on different
//     warps as a skewed wavefront: strip s+1 trails strip s by a few columns and receives the
//     5-state boundary row through L2 as tagged 32-byte slots (one STG.256 / LDG.256 per column).
//   * inside a strip a lane sweeps target columns left to right and keeps the 5 pair-state
//     values of its R rows in registers; the R query rows (20 emissions + 7 transitions each)
//     are TMA-bulk-staged (cp.async.bulk + mbarrier) into the warp's shared-memory slice and
//     read back as warp-uniform broadcast LDS.128.
//   * target operands stream from a JOB-INTERLEAVED copy of the job's column records,
//     [column][k = 0..6][lane] float4 (built per plan by k_interleave_cols), so each of the 7 loads of a
//     column is ONE coalesced 512-byte warp request (4 L1TEX wavefronts instead of 32 when every lane
//     reads its own 112-byte record), register-prefetched one column ahead.
//   * 1 backtrace byte per cell, packed 4 rows per 32-bit word and stored lane-interleaved so
//     every warp store writes one full 128-byte line.
// Arithmetic is the reference's, operation for operation (unfused fp32 mul/add in the same order,
// strict '>' tie rules), so scores and backtrace bytes are bit-identical to the AVX2 (no-FMA) build.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#ifndef HHG_MAX3
#define HHG_MAX3 1   // MM-state maximum as 3-input maxima + equality selects (same bits, fewer ALU-pipe instructions)
#endif

#include "hhg_math.cuh"

namespace hhg {

constexpr int kWarpsPerCta = 4;

struct __align__(16) ColRec {      // one profile column = operands of DP cell (., j)   (112 B)
  float p[20];
  float m2m, m2d, d2m, d2d, i2m;   // tr[j-1][M2M,M2D,D2M,D2D,I2M]
  float i2i, m2i;                  // tr[j][I2I,M2I]
  uint32_t ss;                     // ss_pred*11+ss_conf of column j
};
static_assert(sizeof(ColRec) == 112, "ColRec must be 7 x 16 bytes");

// Boundary hand-off between consecutive strips of a job: the 5 pair-state values of the strip's last
// row at one column plus a tag, written with ONE 256-bit store (sm_100 STG.256 = one 32-byte sector)
// and read with ONE 256-bit L2 load.  The consumer lane re-reads until the tag names the producing
// strip of this run: per-lane dataflow synchronisation with no fences, flags or L1 invalidations.
struct __align__(32) BndSlot {
  float mm, dg, mi, gd, im;
  uint32_t tag;
  uint32_t pad0, pad1;
};
static_assert(sizeof(BndSlot) == 32, "BndSlot must be one 32-byte sector");

// The tag is stored three times (tag, ~tag in pad0, tag in pad1): a consumer accepts a slot only when all three
// agree, so a torn view of the 32 bytes (PTX does not promise single-copy atomicity of a vector access as a whole,
// sm_100 delivers it as one sector transaction) is detected and simply re-read instead of being consumed.
__device__ __forceinline__ void st_slot(BndSlot* p, float mm, float dg, float mi, float gd, float im,
                                        uint32_t tag) {
  asm volatile("st.relaxed.gpu.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p),
               "r"(__float_as_uint(mm)), "r"(__float_as_uint(dg)), "r"(__float_as_uint(mi)),
               "r"(__float_as_uint(gd)), "r"(__float_as_uint(im)), "r"(tag), "r"(~tag), "r"(tag)
               : "memory");
}
// pad0/pad1 are returned so the caller can keep their registers live until the slot is consumed: a dead
// destination register of an in-flight load gets reused by ptxas and the re-use then stalls on the load
// (write-after-write on the long scoreboard; ncu showed 12% of all stall samples on one such FMUL).
__device__ __forceinline__ void ld_slot(const BndSlot* p, float& mm, float& dg, float& mi, float& gd,
                                        float& im, uint32_t& tag, uint32_t& x, uint32_t& y) {
  uint32_t a, b, c, d, e;
  asm volatile("ld.relaxed.gpu.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a), "=r"(b), "=r"(c), "=r"(d), "=r"(e), "=r"(tag), "=r"(x), "=r"(y)
               : "l"(p)
               : "memory");
  mm = __uint_as_float(a); dg = __uint_as_float(b); mi = __uint_as_float(c);
  gd = __uint_as_float(d); im = __uint_as_float(e);
}
// slot valid for tag t: tag == t, pad0 == ~t, pad1 == t
__device__ __forceinline__ bool slot_ok(uint32_t tag, uint32_t pad0, uint32_t pad1, uint32_t want) {
  return ((tag ^ want) | (pad0 ^ ~want) | (pad1 ^ want)) == 0u;
}

struct VitParams {
  // queries: a plan may hold several (query-batch mode, hhblits_omp semantics); every job belongs to one of them
  const float4* qrec;        // query row records (rows 1..Lq of every query, each block zero padded to a multiple of 48)
  const int* job_Lq;         // [njobs] length of the job's query
  const int* job_nstrips;    // [njobs] ceil(Lq / R)
  const int* job_qrow0;      // [njobs] first row record of the job's query in qrec
  const long long* job_ss_off;   // [njobs] offset (in 32-lane blocks) of the job's per-strip maxima
  const int2* items;         // [n_items] work items (job, strip) in dispatch order (see plan_build)
  int n_items;
  // database shard
  const int* Lt;             // [n_targets]
  // plan: the job-interleaved operand stream, [job][column 1..Lmax][k 0..6][lane] float4 (lanes shorter than
  // the job repeat their last column; the cells computed there are never used)
  const float4* jcols;
  const long long* job_jc_off;   // [njobs] offset (in float4) of the job's stream
  // plan
  int njobs;
  const int* job_target;     // [njobs*32] target id (padded lanes repeat a valid id)
  const int* job_Lmax;       // [njobs]
  const long long* job_bt_off;   // [njobs] offset (in uint32 words) into bt
  const long long* job_bnd_off;  // [njobs] offset (in slots) into bnd
  uint32_t* bt;              // packed backtrace words
  struct BndSlot* bnd;       // boundary hand-off slots [job][col][lane], 32 B each (see BndSlot)
  uint32_t tag_base;         // run epoch << 12; slot tag = tag_base + strip + 1
  unsigned int* counter;     // work-item queue head
  float* strip_score;        // [njobs*nstrips*32]
  int* strip_ij;             // [njobs*nstrips*32]  (i<<16 | j)
  const uint32_t* celloff;   // [sum over jobs nstrips*(Lmax+1)*32] bit r = row i0+1+r off, or null
  const long long* job_co_off;
  const float* S33;          // [44*44] or null
  // scoring
  float egq, egt, shift, ssw;
  unsigned long long one2;   // bit pattern of (1.0f, 1.0f); see add2()
  uint32_t zero;             // always 0, opaque to the compiler (register-liveness anchor)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// log2f4 (src/hhutil-inl.h:509-541), degree-4 minimax, unfused.  The sign bit of x must be clear: the reference
// masks it off (i & 0x7F800000), this version does not (ptxas folds the shift and the OR below into one LEA.HI;
// a mask costs an instruction per cell).  dot20_dev never returns a value with the sign bit set.
// The exponent int->float conversion uses the exact magic-number form (no I2F on the hot path):
// bits(8388608.0f) + eb is the float 8388608+eb; subtracting 8388735 (=2^23+127) is exact.
__device__ __forceinline__ float log2f4_dev(float x) {
  const uint32_t u = __float_as_uint(x);
  const float e = __fadd_rn(__uint_as_float((u >> 23) | 0x4B000000u), -8388735.0f);
  const float m = __uint_as_float((u & 0x007FFFFFu) | 0x3F800000u);
  float p = -0.107254423828329604454f;
  p = __fadd_rn(__fmul_rn(p, m), 0.688243882994381274313f);
  p = __fadd_rn(__fmul_rn(p, m), -1.75647175389045657003f);
  p = __fadd_rn(__fmul_rn(p, m), 2.61761038894603480148f);
  p = __fmul_rn(p, __fadd_rn(m, -1.0f));
  return __fadd_rn(p, e);
}

// ScalarProd20Vec (src/hhviterbi.h:126-190) with packed f32x2 arithmetic: the four partial sums
// r0..r3 live in two f32x2 registers (r0,r1) and (r2,r3); each half is an IEEE fp32 mul / add with
// round-to-nearest, i.e. exactly the reference's unfused sequence.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// Packed add as fma(a, ONE, b) with ONE = (1.0f,1.0f) taken from a kernel parameter.  ptxas (12.9)
// contracts a mul.rn.f32x2 feeding an add.rn.f32x2 into one FFMA2 even with -fmad=false, which would
// change the rounding w.r.t. the reference; a*1+b rounds exactly like a+b and, because the value of
// ONE is opaque to the compiler, cannot be folded back into an add and fused.
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b,
                                                   unsigned long long one) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(one), "l"(b));
  return r;
}

// t: 10 packed pairs of the target column, q: float4 x5 of the query row
__device__ __forceinline__ float dot20_dev(const unsigned long long (&t)[10], const float4 (&q)[5],
                                           const unsigned long long one) {
  unsigned long long a01 = mul2(t[0], pack2(q[0].x, q[0].y));
  unsigned long long a23 = mul2(t[1], pack2(q[0].z, q[0].w));
#pragma unroll
  for (int m = 1; m < 5; ++m) {
    a01 = add2(mul2(t[2 * m], pack2(q[m].x, q[m].y)), a01, one);
    a23 = add2(mul2(t[2 * m + 1], pack2(q[m].z, q[m].w)), a23, one);
  }
  float r0, r1, r2, r3;
  unpack2(a01, r0, r1);
  unpack2(a23, r2, r3);
  // |.| on both halves (free FADD operand modifiers): emissions are >= 0 (the C-ABI refuses negative ones), so this
  // changes only a -0.0 sum, from columns of -0.0 emissions, into +0.0, where the reference's log2f4 gives -127
  return __fadd_rn(fabsf(__fadd_rn(r0, r1)), fabsf(__fadd_rn(r2, r3)));
}

// one 16-byte operand of the job-interleaved stream: L2-only load (a line is read once per strip and SM; an L2
// evict_last policy on these loads was measured and changes nothing, profiles/r2_probe_max3_groupsize_dram.txt)
__device__ __forceinline__ float4 ld_jc(const float4* p) { return __ldcg(p); }

#define HHG_NEG (-FLT_MAX)

// ---------------------------------------------------------------------------------------------
// Forward pass.  R rows per strip (multiple of 4).  LOCAL: par.loc.  SS: PRED_PRED ss term.
// CELLOFF: cell-off bit input (alternative alignments / excluded regions).
// ---------------------------------------------------------------------------------------------
template <int R, bool LOCAL, bool SS, bool CELLOFF>
__global__ void __launch_bounds__(kWarpsPerCta * 32, (R <= 12) ? 3 : 2)   // 168 / 255 registers; more resident warps = spills: 9 warps at 224 registers 164 GCUPS, 10 at 200: 122
    k_viterbi(const VitParams P) {
  static_assert(R % 4 == 0, "R must be a multiple of 4");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // smem carve-up: [warps][R] query records | mbarriers | (SS) the S33 table
  float4* qs = reinterpret_cast<float4*>(smem_raw) + (size_t)warp * R * 7;
  constexpr size_t kBarOff = (size_t)kWarpsPerCta * R * 112;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + kBarOff);
  float* s33 = reinterpret_cast<float*>(smem_raw + kBarOff + 64);
  uint64_t* bar = bars + warp;

  if (lane == 0) mbar_init(bar, 1);
  if (SS) {
    for (int k = threadIdx.x; k < 44 * 44; k += blockDim.x) s33[k] = P.S33[k];
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const float smin = LOCAL ? 0.0f : HHG_NEG;
  const int total_items = P.n_items;
  uint32_t parity = 0;

  for (;;) {
    int item = 0;
    if (lane == 0) item = (int)atomicAdd(P.counter, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= total_items) break;
    // the item table is ordered group by group; inside a group of G jobs strip-major, so the strips s and s+1 of
    // one job are dispatched G items apart (natural skew) while the group's targets stay L2-resident
    const int2 it = __ldg(P.items + item);
    const int job = it.x, s = it.y;
    const int Lq = P.job_Lq[job];
    const int nstrips = P.job_nstrips[job];
    const int i0 = s * R;

    // ---- stage this strip's query rows with one TMA bulk copy
    if (lane == 0) {
      mbar_expect_tx(bar, R * 112);
      tma_bulk_g2s(qs, P.qrec + (size_t)(P.job_qrow0[job] + i0) * 7, R * 112, bar);
    }

    const int t = P.job_target[job * 32 + lane];
    const int Lt = P.Lt[t];
    const int Lmax = P.job_Lmax[job];
    const float4* jc = P.jcols + P.job_jc_off[job] + lane;   // operand k of column j: jc[((j-1)*7+k)*32]
    uint32_t* btj = P.bt + P.job_bt_off[job] + lane;
    const size_t bt_row_stride = (size_t)(Lmax + 1) * 32;   // words per 4-row group
    BndSlot* bnd = P.bnd + P.job_bnd_off[job] + lane;
    const uint32_t tag_in = P.tag_base + (uint32_t)s;        // written by strip s-1
    const uint32_t tag_out = P.tag_base + (uint32_t)s + 1u;  // what this strip writes
    const bool last_strip = (s == nstrips - 1);
    const uint32_t* co = nullptr;
    if (CELLOFF) co = P.celloff + P.job_co_off[job] + (size_t)s * (Lmax + 1) * 32 + lane;

    // ---- state of the R rows at the previous column (column 0 initially), :161-173
    float MM[R], GD[R], IM[R], DG[R], MI[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      MM[r] = __fmul_rn((float)(-(i0 + 1 + r)), P.egq);
      GD[r] = IM[r] = DG[r] = MI[r] = HHG_NEG;
    }
    // boundary row i0 at column j-1 (diagonal of the strip's first row)
    float dtMM = __fmul_rn((float)(-i0), P.egq), dtDG = HHG_NEG, dtMI = HHG_NEG, dtGD = HHG_NEG,
          dtIM = HHG_NEG;

    float best = HHG_NEG;
    int bi = 0, bj = 0;

    // first column (register prefetch, one column ahead); L2-only loads: a line is read once per strip
    float4 nx[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) nx[k] = ld_jc(jc + k * 32);   // Lmax >= 1

    // boundary values of column 1 (strips > 0): issue the slot load now, validate the tag at use
    float nMM = 0.f, nDG = 0.f, nMI = 0.f, nGD = 0.f, nIM = 0.f;
    uint32_t ntag = 0, npad0 = 0, npad1 = 0;
    if (s > 0) ld_slot(bnd + 32, nMM, nDG, nMI, nGD, nIM, ntag, npad0, npad1);

    mbar_wait(bar, parity);
    parity ^= 1u;

    for (int j = 1; j <= Lmax; ++j) {
      // ---- current column operands (from the prefetch registers), prefetch the next column
      unsigned long long tp[10];
      tp[0] = pack2(nx[0].x, nx[0].y); tp[1] = pack2(nx[0].z, nx[0].w);
      tp[2] = pack2(nx[1].x, nx[1].y); tp[3] = pack2(nx[1].z, nx[1].w);
      tp[4] = pack2(nx[2].x, nx[2].y); tp[5] = pack2(nx[2].z, nx[2].w);
      tp[6] = pack2(nx[3].x, nx[3].y); tp[7] = pack2(nx[3].z, nx[3].w);
      tp[8] = pack2(nx[4].x, nx[4].y); tp[9] = pack2(nx[4].z, nx[4].w);
      const float t_m2m = nx[5].x, t_m2d = nx[5].y, t_d2m = nx[5].z, t_d2d = nx[5].w;
      const float t_i2m = nx[6].x, t_i2i = nx[6].y, t_m2i = nx[6].z;
      const uint32_t t_ss = __float_as_uint(nx[6].w);
      {
        const float4* src = jc + (size_t)(min(j + 1, Lmax) - 1) * 224;
#pragma unroll
        for (int k = 0; k < 7; ++k) nx[k] = ld_jc(src + k * 32);
      }

      // ---- boundary row i0 at column j: slot prefetched during column j-1; spin (per lane) until the
      // producer strip's tag is there, then prefetch column j+1
      float tMM, tDG, tMI, tGD, tIM;
      if (s == 0) {
        tMM = __fmul_rn((float)(-j), P.egt);   // :148
        tDG = tMI = tGD = tIM = HHG_NEG;
      } else {
        // all three copies of the tag must agree (also keeps the pad registers live, see ld_slot)
        while (!slot_ok(ntag, npad0, npad1, tag_in)) {
          __nanosleep(20);
          ld_slot(bnd + (size_t)j * 32, nMM, nDG, nMI, nGD, nIM, ntag, npad0, npad1);
        }
        tMM = nMM; tDG = nDG; tMI = nMI; tGD = nGD; tIM = nIM;
        if (j < Lmax) ld_slot(bnd + (size_t)(j + 1) * 32, nMM, nDG, nMI, nGD, nIM, ntag, npad0, npad1);
      }
      uint32_t cow = 0;
      if (CELLOFF) cow = __ldg(co + (size_t)j * 32);

      float dMM = dtMM, dGD = dtGD, dIM = dtIM, dDG = dtDG, dMI = dtMI;   // cell (i-1, j-1)
      float uMM = tMM, uDG = tDG, uMI = tMI;                              // cell (i-1, j)
      const float bcmp = (j <= Lt) ? best : INFINITY;   // padded columns never become the maximum
      float bc = bcmp;

      // (t_ss & P.zero) is 0; it only keeps the 4th register of the prefetch LDG.128 live (see ld_slot)
      uint32_t word = SS ? 0u : (t_ss & P.zero);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        float4 q[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) q[k] = qs[r * 7 + k];
        const float4 qa = qs[r * 7 + 5], qb = qs[r * 7 + 6];
        const float q_m2m = qa.x, q_m2d = qa.y, q_d2m = qa.z, q_d2d = qa.w;
        const float q_i2m = qb.x, q_i2i = qb.y, q_m2i = qb.z;

        const float oMM = MM[r], oGD = GD[r], oIM = IM[r], oDG = DG[r], oMI = MI[r];   // (i, j-1)

        // 5-way maximum with the reference's strict-'>' / first-wins rule, :241-273
        uint32_t b;
        float mm;
        const float c1 = __fadd_rn(__fadd_rn(dMM, q_m2m), t_m2m);
        const float c2 = __fadd_rn(__fadd_rn(dGD, q_m2m), t_d2m);
        const float c3 = __fadd_rn(__fadd_rn(dIM, q_i2m), t_m2m);
        const float c4 = __fadd_rn(__fadd_rn(dDG, q_d2m), t_m2m);
        const float c5 = __fadd_rn(__fadd_rn(dMI, q_m2m), t_i2m);
#if HHG_MAX3
        // the winner of the strict-'>' chain is the FIRST candidate (order STOP, MM, GD, IM, DG, MI) that attains
        // the maximum: three 3-input maxima (FMNMX3) + five equality selects instead of five max + five '>' selects
        mm = fmaxf(fmaxf(smin, c1), c2);
        mm = fmaxf(fmaxf(mm, c3), c4);
        mm = fmaxf(mm, c5);
        b = 6u;
        b = (c4 == mm) ? 5u : b;
        b = (c3 == mm) ? 4u : b;
        b = (c2 == mm) ? 3u : b;
        b = (c1 == mm) ? 2u : b;
        b = (smin == mm) ? 0u : b;
#else
        b = (c1 > smin) ? 2u : 0u; mm = fmaxf(smin, c1);
        b = (c2 > mm) ? 3u : b;    mm = fmaxf(mm, c2);
        b = (c3 > mm) ? 4u : b;    mm = fmaxf(mm, c3);
        b = (c4 > mm) ? 5u : b;    mm = fmaxf(mm, c4);
        b = (c5 > mm) ? 6u : b;    mm = fmaxf(mm, c5);
#endif

        float Si = log2f4_dev(dot20_dev(tp, q, P.one2));                       // :277
        if (SS) {
          const uint32_t q_ss = __float_as_uint(qb.w);
          Si = __fadd_rn(__fmul_rn(P.ssw, s33[q_ss * 44 + t_ss]), Si);   // :210,279
        }
        Si = __fadd_rn(Si, P.shift);                                   // :281
        mm = __fadd_rn(mm, Si);

        float a1, a2, gd, im, dg, mi;
        a1 = __fadd_rn(oMM, t_m2d); a2 = __fadd_rn(oGD, t_d2d);                                // :307
        b |= (a1 > a2) ? 8u : 0u;  gd = fmaxf(a1, a2);
        a1 = __fadd_rn(__fadd_rn(oMM, q_m2i), t_m2m); a2 = __fadd_rn(__fadd_rn(oIM, q_i2i), t_m2m);   // :324
        b |= (a1 > a2) ? 16u : 0u; im = fmaxf(a1, a2);
        a1 = __fadd_rn(uMM, q_m2d); a2 = __fadd_rn(uDG, q_d2d);                                // :340
        b |= (a1 > a2) ? 32u : 0u; dg = fmaxf(a1, a2);
        a1 = __fadd_rn(__fadd_rn(uMM, q_m2m), t_m2i); a2 = __fadd_rn(__fadd_rn(uMI, q_m2m), t_i2i);   // :358
        b |= (a1 > a2) ? 64u : 0u; mi = fmaxf(a1, a2);

        if (CELLOFF) {                                                 // :373-392
          const float off = ((cow >> r) & 1u) ? HHG_NEG : 0.0f;
          mm = __fadd_rn(mm, off); gd = __fadd_rn(gd, off); im = __fadd_rn(im, off);
          dg = __fadd_rn(dg, off); mi = __fadd_rn(mi, off);
        }

        word |= b << (8 * (r & 3));
        if ((r & 3) == 3) {
          __stcs(btj + (size_t)((i0 >> 2) + (r >> 2)) * bt_row_stride + (size_t)j * 32, word);
          word = 0;
        }
        // rotate: this row's old values are the next row's diagonal, its new values the next row's up
        dMM = oMM; dGD = oGD; dIM = oIM; dDG = oDG; dMI = oMI;
        uMM = mm; uDG = dg; uMI = mi;
        MM[r] = mm; GD[r] = gd; IM[r] = im; DG[r] = dg; MI[r] = mi;
      }
      dtMM = tMM; dtDG = tDG; dtMI = tMI; dtGD = tGD; dtIM = tIM;

      // running maximum, :423-455: ONE test per column on the maximum of the R new MM values (a tree of
      // FMNMX, 1 instruction per row instead of compare+branch per cell); only when it can matter the
      // rows are examined in ascending order.  Strips are swept column-major, the reference row-major:
      // on an exact tie the earlier ROW must win (mm == best && i < bi).
      {
        float cm[R];
#pragma unroll
        for (int r = 0; r < R; ++r) cm[r] = MM[r];
#pragma unroll
        for (int n = R; n > 1; n = (n + 1) / 2) {      // pairwise tree, any R
#pragma unroll
          for (int r = 0; r < n / 2; ++r) cm[r] = fmaxf(cm[r], cm[r + (n + 1) / 2]);
        }
        if (cm[0] >= bc) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const float mm = MM[r];
            if (mm >= bc) {
              const int i = i0 + 1 + r;
              const bool cand = (i <= Lq) && (LOCAL || i == Lq || j == Lt);
              if (cand && (mm > best || i < bi)) { best = mm; bi = i; bj = j; bc = mm; }
            }
          }
        }
      }

      if (!last_strip)
        st_slot(bnd + (size_t)j * 32, MM[R - 1], DG[R - 1], MI[R - 1], GD[R - 1], IM[R - 1], tag_out);
    }
    const size_t o = ((size_t)P.job_ss_off[job] + s) * 32 + lane;
    P.strip_score[o] = best;
    P.strip_ij[o] = (bi << 16) | bj;
    __syncwarp();   // all lanes done with the smem slice before the next TMA overwrites it
  }
}

// pnul[a] of HMM::IncludeNullModelInHMM (src/hhhmm.cpp:2059-2088) for one (query, template) pair.
// columnscore: 0 = pb, 1 = 0.5(q.pav + t.pav) (default), 2 = t.pav, 3 = q.pav.
__device__ __forceinline__ void null_model_vec(int columnscore, const float* __restrict__ q_pav,
                                               const float* __restrict__ t_pav, const float* __restrict__ pb,
                                               float (&pn)[20]) {
#pragma unroll
  for (int a = 0; a < 20; ++a) {
    switch (columnscore) {
      case 0: pn[a] = pb[a]; break;
      case 2: pn[a] = t_pav[a]; break;
      case 3: pn[a] = q_pav[a]; break;
      default: pn[a] = __fmul_rn(0.5f, __fadd_rn(q_pav[a], t_pav[a])); break;
    }
  }
}
__device__ __forceinline__ float4 div4(float4 v, const float* pn) {
  v.x = __fdiv_rn(v.x, pn[0]); v.y = __fdiv_rn(v.y, pn[1]); v.z = __fdiv_rn(v.z, pn[2]); v.w = __fdiv_rn(v.w, pn[3]);
  return v;
}

// ---------------------------------------------------------------------------------------------
// Backtrace: one thread per requested target.  Merges the per-strip maxima in row order (strict '>',
// i.e. the reference's row-major first-occurrence rule) and walks the packed byte matrix.
// ---------------------------------------------------------------------------------------------
struct HitRec {
  float score;
  int i2, j2, i1, j1, nsteps, matched_cols, path_off;
  float hit_score;   // Hit.score: Viterbi score - ss score + correlation term (src/hhviterbi.cpp:215-256)
  float score_ss;    // Hit.score_ss
};

struct BtParams {
  int n_req;
  const int* job_nstrips;    // [njobs]
  const long long* job_ss_off;
  const int* job_qrow0;      // [njobs] first row record of the job's query
  // fused null model (query-batch plans over a raw shard): cols = emissions BEFORE the null model and the division
  // t.p[j][a] / pnul[a] is applied on the fly exactly like HMM::IncludeNullModelInHMM; nm_mode < 0: cols are prepared
  int nm_mode;
  const int* job_query;      // [njobs]
  const float* q_pav;        // [nq*20]
  const float* t_pav;        // [n_targets*20]
  const float* pb;           // [20]
  int job_begin, job_end;    // only requests whose job lies in [job_begin, job_end) are traced
  const int* req_job;        // [n_req]
  const int* req_lane;       // [n_req]
  const int* job_Lmax;
  const long long* job_bt_off;
  const uint32_t* bt;
  const float* strip_score;
  const int* strip_ij;
  const long long* path_off; // [n_req] offsets into paths
  HitRec* hits;
  uint8_t* paths;            // may be null
  // Hit.score (Viterbi::ScoreForBacktrace, src/hhviterbi.cpp:195-281)
  const int* req_target;     // [n_req] target id in the shard
  const float4* qrec;        // query row records (p in the first 5 float4)
  const float4* cols;        // target column records
  const long long* col_off;
  const float* lg2;          // fast_log2 tables (src/util-inl.h:108-128): lg2[1025], diff[1025]
  const float* diff;
  const float* S33;          // may be null
  float* S;                  // [path_total] per-step column scores (scratch)
  float corr, ssw;
  int use_ss;                // PRED_PRED ss term was part of the alignment score
  int ss_score_mode;         // par.ssm == 2: subtract the ss score again (SCORE_ALIGNMENT)
};

// Score(q.p[i], t.p[j]) = fast_log2(ScalarProd20(q, t)), src/hhhit-inl.h:61-134.  In the AVX2 build of the
// reference (the pinned oracle) the macro SSE is not defined in that header, so ScalarProd20 is the
// plain left-to-right sum  t0*q0 + t1*q1 + ... + t19*q19  (verified against the compiled reference:
// 300/300 random vectors bit-identical; the SSE shuffle tree matches only ~70%).
__device__ __forceinline__ float score_cols_dev(const float4* q, const float4* t, const float* lg2,
                                                const float* diff, const float* pn = nullptr) {
  float sum = 0.0f;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const float4 a = q[k];
    const float4 b = pn ? div4(t[k], pn + 4 * k) : t[k];
    if (k == 0) sum = __fmul_rn(b.x, a.x); else sum = __fadd_rn(sum, __fmul_rn(b.x, a.x));
    sum = __fadd_rn(sum, __fmul_rn(b.y, a.y));
    sum = __fadd_rn(sum, __fmul_rn(b.z, a.z));
    sum = __fadd_rn(sum, __fmul_rn(b.w, a.w));
  }
  return fast_log2_dev(sum, lg2, diff);
}

__device__ __forceinline__ uint32_t bt_byte(const uint32_t* btj, size_t row_stride, int i, int j) {
  const uint32_t w = btj[(size_t)((i - 1) >> 2) * row_stride + (size_t)j * 32];
  return (w >> (8 * ((i - 1) & 3))) & 0xFFu;
}

__global__ void k_backtrace(const BtParams P) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= P.n_req) return;
  const int job = P.req_job[k], lane = P.req_lane[k];
  if (job < P.job_begin || job >= P.job_end) return;
  float best = HHG_NEG;
  int ij = 0;
  const int nstrips = P.job_nstrips[job];
  for (int s = 0; s < nstrips; ++s) {
    const size_t o = ((size_t)P.job_ss_off[job] + s) * 32 + lane;
    const float v = P.strip_score[o];
    if (v > best) { best = v; ij = P.strip_ij[o]; }
  }
  const int i2 = ij >> 16, j2 = ij & 0xFFFF;
  const int Lmax = P.job_Lmax[job];
  const uint32_t* btj = P.bt + P.job_bt_off[job] + lane;
  const size_t rs = (size_t)(Lmax + 1) * 32;
  uint8_t* path = P.paths ? P.paths + P.path_off[k] : nullptr;

  const float4* tcol = P.cols + (size_t)P.col_off[P.req_target[k]] * 7;
  const float4* qrec = P.qrec + (size_t)P.job_qrow0[job] * 7;
  float pnv[20];
  const float* pn = nullptr;
  if (P.nm_mode >= 0) {
    null_model_vec(P.nm_mode, P.q_pav + (size_t)P.job_query[job] * 20, P.t_pav + (size_t)P.req_target[k] * 20, P.pb, pnv);
    pn = pnv;
  }
  float* S = P.S + P.path_off[k];
  float score_ss = 0.0f;

  int step = 0, i = i2, j = j2, mc = 0, li = i2, lj = j2;
  int state = 2;   // MM
  while (state != 0) {
    if (path) path[step] = (uint8_t)state;
    // per-step column score: only MM steps score (src/hhviterbi.cpp:219-235); the step that turns out to
    // be the last one is re-scored below because the reference forces states[nsteps] = MM first
    float Sv = 0.0f;
    if (state == 2 && i >= 1 && j >= 1) {
      Sv = score_cols_dev(qrec + (size_t)(i - 1) * 7, tcol + (size_t)(j - 1) * 7, P.lg2, P.diff, pn);
      if (P.use_ss) {
        const uint32_t qs = __float_as_uint(qrec[(size_t)(i - 1) * 7 + 6].w);
        const uint32_t ts = __float_as_uint(tcol[(size_t)(j - 1) * 7 + 6].w);
        score_ss = __fadd_rn(score_ss, __fmul_rn(P.ssw, P.S33[qs * 44 + ts]));
      }
    }
    S[step] = Sv;
    ++step;
    li = i; lj = j;
    const uint32_t c = (i >= 1 && j >= 1) ? bt_byte(btj, rs, i, j) : 0u;
    const int prev_state = state;
    switch (state) {
      case 2: ++mc; state = (i <= 1 || j <= 1) ? 0 : (int)(c & 7u); --i; --j; break;
      case 3: if (j <= 1) state = 0; else { if (c & 8u) state = 2; --j; } break;
      case 4: if (j <= 1) state = 0; else { if (c & 16u) state = 2; --j; } break;
      case 5: if (i <= 1) state = 0; else { if (c & 32u) state = 2; --i; } break;
      case 6: if (i <= 1) state = 0; else { if (c & 64u) state = 2; --i; } break;
      default: state = 0; break;
    }
    if (state == 0 && prev_state != 2 && li >= 1 && lj >= 1) {
      // last step ended in a gap state: the reference relabels it MM (src/hhviterbi.cpp:147) and scores it
      S[step - 1] = score_cols_dev(qrec + (size_t)(li - 1) * 7, tcol + (size_t)(lj - 1) * 7, P.lg2, P.diff, pn);
      if (P.use_ss) {
        const uint32_t qs = __float_as_uint(qrec[(size_t)(li - 1) * 7 + 6].w);
        const uint32_t ts = __float_as_uint(tcol[(size_t)(lj - 1) * 7 + 6].w);
        score_ss = __fadd_rn(score_ss, __fmul_rn(P.ssw, P.S33[qs * 44 + ts]));
      }
    }
  }
  if (path && step > 0) path[step - 1] = 2;   // states[nsteps] = MM, src/hhviterbi.cpp:147
  // Hit.score, src/hhviterbi.cpp:237-256: four correlation passes in the reference's order
  float hs = best;
  if (P.ss_score_mode) hs = __fadd_rn(hs, -score_ss);
  float scorr = 0.0f;
  if (step > 0) {
    for (int d = 1; d <= 4; ++d)
      for (int st = d; st < step; ++st) scorr = __fadd_rn(scorr, __fmul_rn(S[st], S[st - d]));
    hs = __fadd_rn(hs, __fmul_rn(P.corr, scorr));
  }
  HitRec h;
  h.score = best; h.i2 = i2; h.j2 = j2; h.i1 = li; h.j1 = lj; h.nsteps = step;
  h.matched_cols = mc; h.path_off = (int)P.path_off[k];
  h.hit_score = hs; h.score_ss = score_ss;
  P.hits[k] = h;
}

// Query-dependent part of PrepareTemplateHMM: factor the null model into the template emissions
// (HMM::IncludeNullModelInHMM, src/hhhmm.cpp:2059-2088).  One thread per target column; exact fp32
// division like the reference.  columnscore: 0 = pb, 1 = 0.5(q.pav + t.pav) (default), 2 = t.pav, 3 = q.pav.
__global__ void k_null_model(long long total_cols, int n, const long long* col_off, const float4* raw,
                             const float* t_pav, const float* q_pav, const float* pb, int columnscore,
                             float4* out) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= total_cols) return;
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (col_off[mid] <= c) lo = mid; else hi = mid - 1;
  }
  float pn[20];
  null_model_vec(columnscore, q_pav, t_pav + (size_t)lo * 20, pb, pn);
  const float4* src = raw + (size_t)c * 7;
  float4* dst = out + (size_t)c * 7;
#pragma unroll
  for (int k = 0; k < 5; ++k) dst[k] = div4(src[k], pn + 4 * k);
  dst[5] = src[5];
  dst[6] = src[6];
}

// Compact the per-request path strings (capacity Lq+Lt+2 each) to their real lengths before the D2H copy:
// one thread per request copies nsteps bytes to its compact offset.
__global__ void k_gather_paths(int n, const HitRec* hits, const long long* src_off, const long long* dst_off,
                               const uint8_t* src, uint8_t* dst) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int len = hits[k].nsteps;
  const uint8_t* s = src + src_off[k];
  uint8_t* d = dst + dst_off[k];
  for (int b = 0; b < len; ++b) d[b] = s[b];
}

// De-interleave one target's backtrace bytes into the reference's row-major cell matrix (parity tests).
__global__ void k_debug_bt(const uint32_t* bt, long long bt_off, int lane, int Lmax, int Lq, int Lt,
                           uint8_t* out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = (Lq + 1) * (Lt + 1);
  if (idx >= total) return;
  const int i = idx / (Lt + 1), j = idx - i * (Lt + 1);
  uint8_t v = 0;
  if (i >= 1 && j >= 1) v = (uint8_t)bt_byte(bt + bt_off + lane, (size_t)(Lmax + 1) * 32, i, j);
  out[idx] = v;
}

// Pack prepared profiles (include/hhg.h layout) into column records: thread per (target, column).
__global__ void k_pack_cols(int n, const int* L, const long long* col_off, const long long* p_off,
                            const long long* tr_off, const long long* ss_off, const float* p,
                            const float* tr, const uint8_t* ss, ColRec* out, long long total_cols) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= total_cols) return;
  // binary search the target owning column c
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (col_off[mid] <= c) lo = mid; else hi = mid - 1;
  }
  const int t = lo;
  const int j = (int)(c - col_off[t]) + 1;   // 1-based column
  const float* pp = p + p_off[t] + (size_t)j * 20;
  const float* t1 = tr + tr_off[t] + (size_t)(j - 1) * 7;
  const float* t0 = tr + tr_off[t] + (size_t)j * 7;
  ColRec r;
#pragma unroll
  for (int a = 0; a < 20; ++a) r.p[a] = pp[a];
  r.m2m = t1[0]; r.m2d = t1[2]; r.d2m = t1[5]; r.d2d = t1[6]; r.i2m = t1[3];
  r.i2i = t0[4]; r.m2i = t0[1];
  r.ss = ss ? (uint32_t)ss[ss_off[t] + j] : 0u;
  out[c] = r;
}

// Build the job-interleaved operand stream of a plan from the shard's column records: warp per (job, column),
// lane = the job's lane.  Each lane copies its own 112-byte record (7 x 16 B) of column min(j, Lt) into
// out[job_jc_off[job] + ((j-1)*7 + k)*32 + lane]: the seven stores of a warp are full 512-byte lines.
__global__ void __launch_bounds__(256)
k_interleave_cols(int njobs, const int* __restrict__ job_target, const int* __restrict__ job_Lmax,
                  const long long* __restrict__ job_jc_off, const float4* __restrict__ cols,
                  const long long* __restrict__ col_off, const int* __restrict__ Lt, float4* __restrict__ out,
                  int nm_mode, const int* __restrict__ job_query, const float* __restrict__ q_pav,
                  const float* __restrict__ t_pav, const float* __restrict__ pb) {
  const int job = blockIdx.x;
  const int lane = threadIdx.x & 31;
  const int Lmax = job_Lmax[job];
  const int t = job_target[job * 32 + lane];
  const int L = Lt[t];
  const float4* src0 = cols + (size_t)col_off[t] * 7;
  float4* dst0 = out + job_jc_off[job] + lane;
  // nm_mode >= 0: `cols` holds the emissions before the null model; factor it in for this job's query on the way
  // (HMM::IncludeNullModelInHMM, the query-dependent step of PrepareTemplateHMM), so a batch of queries can share one
  // resident raw shard
  float pn[20];
  if (nm_mode >= 0) null_model_vec(nm_mode, q_pav + (size_t)job_query[job] * 20, t_pav + (size_t)t * 20, pb, pn);
  for (int j = blockIdx.y * 8 + (threadIdx.x >> 5) + 1; j <= Lmax; j += gridDim.y * 8) {
    const float4* src = src0 + (size_t)(min(j, L) - 1) * 7;
    float4* dst = dst0 + (size_t)(j - 1) * 224;
#pragma unroll
    for (int k = 0; k < 5; ++k) dst[k * 32] = nm_mode >= 0 ? div4(__ldg(src + k), pn + 4 * k) : __ldg(src + k);
    dst[5 * 32] = __ldg(src + 5);
    dst[6 * 32] = __ldg(src + 6);
  }
}

// Rasterise excluded alignments into the cell-off bit words (Viterbi::ExcludeAlignment,
// src/hhviterbi.cpp:61-77): one thread per excluded path step.
__global__ void k_celloff_raster(int n_steps, const int* step_req, const int* step_i, const int* step_j,
                                 const int* req_job, const int* req_lane, const int* req_Lt, const int* req_Lq,
                                 const int* job_Lmax, const long long* job_co_off, int R,
                                 uint32_t* co) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_steps) return;
  const int rq = step_req[k];
  const int job = req_job[rq], lane = req_lane[rq], Lt = req_Lt[rq], Lq = req_Lq[rq];
  const int Lmax = job_Lmax[job];
  uint32_t* base = co + job_co_off[job] + lane;
  const int i = step_i[k], j = step_j[k];
  const int W = 40;   // VITERBI_PATH_WIDTH, src/hhdecl.h:50
  for (int ii = max(i - W, 1); ii <= min(i + W, Lq); ++ii) {
    const int s = (ii - 1) / R, r = (ii - 1) - s * R;
    atomicOr(base + ((size_t)s * (Lmax + 1) + j) * 32, 1u << r);
  }
  for (int jj = max(j - W, 1); jj <= min(j + W, Lt); ++jj) {
    const int s = (i - 1) / R, r = (i - 1) - s * R;
    atomicOr(base + ((size_t)s * (Lmax + 1) + jj) * 32, 1u << r);
  }
}

// Excluded regions (ViterbiRunner::exclude_regions / exclude_template_regions, src/hhviterbirunner.cpp:291-330; the
// -excl / -template_excl options): query rows i0..i1 are switched off for every template column, template columns
// j0..j1 for every query row.  One thread per cell-off word (job, strip, column, lane).
__global__ void __launch_bounds__(256)
k_celloff_regions(long long n_words, int njobs, const long long* __restrict__ job_co_off, const int* __restrict__ job_Lmax,
                  const int* __restrict__ job_nstrips, int R, int nqr, const int* __restrict__ q_lo,
                  const int* __restrict__ q_hi, int ntr, const int* __restrict__ t_lo, const int* __restrict__ t_hi,
                  uint32_t* __restrict__ co) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  int lo = 0, hi = njobs - 1;                       // job owning word w
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (job_co_off[mid] <= w) lo = mid; else hi = mid - 1;
  }
  const long long rel = w - job_co_off[lo];
  const int cols1 = job_Lmax[lo] + 1;
  const int s = (int)(rel / ((long long)cols1 * 32));
  const int j = (int)((rel / 32) % cols1);
  if (s >= job_nstrips[lo] || j < 1) return;
  uint32_t m = 0;
  for (int k = 0; k < ntr; ++k) if (j >= t_lo[k] && j <= t_hi[k]) m = 0xFFFFFFFFu;
  for (int k = 0; k < nqr && m != 0xFFFFFFFFu; ++k) {
    const int a = max(q_lo[k], s * R + 1), b = min(q_hi[k], s * R + R);   // rows of this strip inside the range
    if (a <= b) m |= (b - a + 1 >= 32 ? 0xFFFFFFFFu : ((1u << (b - a + 1)) - 1u)) << (a - 1 - s * R);
  }
  if (m) co[w] |= m;
}

// ---------------------------------------------------------------------------------------------
// cs219 ungapped prefilter (Prefilter::ungapped_sse_score, src/hhprefilter.cpp:214-275).
//   S(i,j) = max(0, min(255, S(i-1,j-1) + prof[x_j][i]) - offset);  score = max over all cells.
// One warp per database sequence.  The query is cut into TILES of 64*WB positions (WB <= 8, one launch per
// tile, so a query of any length works); inside a tile lane l owns the contiguous positions
// [l*2WB, (l+1)*2WB) as WB registers of two 16-bit values: register w holds position l*2WB + w in its low
// half and l*2WB + WB + w in its high half.  With that pairing the diagonal predecessor of BOTH halves of
// register w is register w-1, so the sweep needs no funnel shifts: one byte-permute per column builds the
// carry into register 0 (low half: last position of lane l-1 via one shuffle, high half: position WB-1 of
// the own lane).  The u8-saturating recurrence is exact in 16-bit integers:
//   min(S + p, 255) - offset = min(S + (p - offset), 255 - offset),  then max(., 0)
// = ONE DPX instruction per two cells, __viaddmin_s16x2_relu(S, p - offset, 255 - offset); the running
// maximum takes one __vimax3_s16x2 per two registers.  The profile (p - offset as s16x2, [state][w][lane]
// words, 28 KB per WB) sits in shared memory; the 32 lanes of a warp read 128 contiguous bytes.
// Tile t > 0 needs S of the previous tile's last position at column j-1: tile t-1 stores that byte per
// column (edge_out), tile t reads it (edge_in); the per-sequence maximum is combined across tiles in `scores`.
// Positions past the end of the query carry p = 0: their S is always < the diagonal predecessor's (or 0) and
// never changes the maximum.
// ---------------------------------------------------------------------------------------------
struct PfParams {
  int n;
  const int* L;
  const long long* off;
  const uint8_t* seq;
  const uint32_t* prof32;   // this tile's profile: [220][WB][32] words (p - offset | p - offset) as s16x2
  int offset;
  int tile, last_tile;      // tile index; 1 if no further tile follows
  const uint8_t* edge_in;   // [sum L] S(last position of tile-1, column) per sequence column (tile > 0)
  uint8_t* edge_out;        // [sum L] written when !last_tile
  int* scores;              // running maximum over the tiles launched so far
  unsigned int* counter;
};

template <int WB>   // 32-bit s16x2 registers per lane: the tile covers 64*WB query positions
__global__ void __launch_bounds__(512) k_prefilter_ungapped(const PfParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint32_t* sprof = reinterpret_cast<uint32_t*>(smem_raw);   // [220][WB][32]
  for (int idx = threadIdx.x; idx < 220 * WB * 32; idx += blockDim.x) sprof[idx] = P.prof32[idx];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const uint32_t cap = (uint32_t)(255 - P.offset) * 0x00010001u;           // 255 - offset | 255 - offset
  const bool first_tile = P.tile == 0;
  for (;;) {
    int n = 0;
    if (lane == 0) n = (int)atomicAdd(P.counter, 1u);
    n = __shfl_sync(0xffffffffu, n, 0);
    if (n >= P.n) break;
    const long long o = P.off[n];
    const uint8_t* x = P.seq + o;
    const int L = P.L[n];
    uint32_t S[WB];
#pragma unroll
    for (int w = 0; w < WB; ++w) S[w] = 0;
    uint32_t smax = 0;
    for (int j0 = 0; j0 < L; j0 += 32) {
      const int xl = (j0 + lane < L) ? (int)x[j0 + lane] : 0;
      // carry into the tile at column j = S(last position of the previous tile, column j-1)
      int el = 0;
      if (!first_tile && j0 + lane >= 1 && j0 + lane <= L) el = (int)P.edge_in[o + j0 + lane - 1];
      const int cnt = min(32, L - j0);
      uint32_t eout = 0;
      for (int jj = 0; jj < cnt; ++jj) {
        const int xs = __shfl_sync(0xffffffffu, xl, jj);
        const uint32_t* prow = sprof + (size_t)xs * (WB * 32) + lane;
        uint32_t up = __shfl_up_sync(0xffffffffu, S[WB - 1], 1);
        const uint32_t ein = first_tile ? 0u : (uint32_t)__shfl_sync(0xffffffffu, el, jj);   // warp-uniform branch
        if (lane == 0) up = ein << 16;
        // register 0's diagonal inputs: low half <- high half of `up` (position l*2WB-1), high half <- low half
        // of the own last register (position l*2WB+WB-1)
        const uint32_t carry = __byte_perm(up, S[WB - 1], 0x5432);
#pragma unroll
        for (int w = WB - 1; w >= 1; --w) S[w] = __viaddmin_s16x2_relu(S[w - 1], prow[w * 32], cap);
        S[0] = __viaddmin_s16x2_relu(carry, prow[0], cap);
#pragma unroll
        for (int w = 0; w + 1 < WB; w += 2) smax = __vimax3_s16x2(smax, S[w], S[w + 1]);
        if (WB & 1) smax = __vimax3_s16x2(smax, S[WB - 1], 0u);
        if (!P.last_tile) {
          // S(last position of this tile, column j0+jj): lane 31, last register, high half; lane jj keeps it
          const uint32_t e = __shfl_sync(0xffffffffu, S[WB - 1] >> 16, 31);
          if (lane == jj) eout = e;
        }
      }
      if (!P.last_tile && lane < cnt) P.edge_out[o + j0 + lane] = (uint8_t)eout;
    }
    uint32_t m = max(smax & 0xFFFFu, smax >> 16);
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, k));
    if (lane == 0) P.scores[n] = first_tile ? (int)m : max(P.scores[n], (int)m);
  }
}

// ---------------------------------------------------------------------------------------------
// Gapped byte Smith-Waterman of prefilter stage 2 (Prefilter::swStripedByte, src/hhprefilter.cpp:70-212).
// The reference's Farrar-striped AVX2 routine has 32 byte lanes and a lazy-F loop that does not update E,
// so its score can depend on the striping (SURVEY App. D-5).  To be bit-identical we execute exactly that
// algorithm: one WARP = the 32 byte lanes of the AVX2 vector (lane k owns query positions k*W + j),
// the full-width byte shift is __shfl_up, the movemask test is __all_sync.  Stage 2 only sees the
// survivors of stage 1 (hundreds..thousands of sequences), so one byte per lane is plenty.
// ---------------------------------------------------------------------------------------------
struct SwParams {
  int n;                    // number of requested sequences
  const int* ids;           // [n] sequence ids (null = 0..n-1)
  const int* L;
  const long long* off;
  const uint8_t* seq;
  const uint8_t* prof;      // striped profile [220][W][32]: byte (k, j, lane) = position lane*W + j (bias pad)
  int W;
  int gap_open, gap_extend, bias;
  int* scores;              // [n]
  unsigned int* counter;
};

template <bool PROF_SMEM>   // false: the striped profile does not fit in shared memory (Lq > ~900) and is read from L2
__global__ void __launch_bounds__(256) k_prefilter_sw(const SwParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int W = P.W;
  const uint8_t* sprof = PROF_SMEM ? smem_raw : P.prof;        // [220][W][32]
  if (PROF_SMEM) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(P.prof);
    uint32_t* dst = reinterpret_cast<uint32_t*>(smem_raw);
    for (int idx = threadIdx.x; idx < 220 * W * 8; idx += blockDim.x) dst[idx] = src[idx];
    __syncthreads();
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* Hst = smem_raw + (PROF_SMEM ? (size_t)220 * W * 32 : 0) + (size_t)warp * 3 * W * 32 + lane;   // + j*32
  uint8_t* Hld = Hst + (size_t)W * 32;
  uint8_t* E = Hld + (size_t)W * 32;
  const int go = P.gap_open, ge = P.gap_extend, bias = P.bias;
  for (;;) {
    int it = 0;
    if (lane == 0) it = (int)atomicAdd(P.counter, 1u);
    it = __shfl_sync(0xffffffffu, it, 0);
    if (it >= P.n) break;
    const int id = P.ids ? P.ids[it] : it;
    const uint8_t* x = P.seq + P.off[id];
    const int L = P.L[id];
    for (int j = 0; j < W; ++j) { Hst[j * 32] = 0; Hld[j * 32] = 0; E[j * 32] = 0; }
    int vmax = 0;
    for (int i = 0; i < L; ++i) {
      int vF = 0, vMaxCol = 0;
      int vH = __shfl_up_sync(0xffffffffu, (int)Hst[(W - 1) * 32], 1);
      if (lane == 0) vH = 0;
      const uint8_t* row = sprof + (size_t)x[i] * W * 32 + lane;
      { uint8_t* t = Hld; Hld = Hst; Hst = t; }
      for (int j = 0; j < W; ++j) {
        int h = min(vH + (int)row[j * 32], 255);
        h = max(h - bias, 0);
        int e = E[j * 32];
        h = max(h, e);
        h = max(h, vF);
        vMaxCol = max(vMaxCol, h);
        Hst[j * 32] = (uint8_t)h;
        h = max(h - go, 0);
        e = max(max(e - ge, 0), h);
        E[j * 32] = (uint8_t)e;
        vF = max(max(vF - ge, 0), h);
        vH = Hld[j * 32];
      }
      // lazy F (:158-196)
      int j = 0;
      vF = __shfl_up_sync(0xffffffffu, vF, 1);
      if (lane == 0) vF = 0;
      for (;;) {
        int h = Hst[j * 32];
        const bool done = max(vF - max(h - go, 0), 0) == 0;
        if (__all_sync(0xffffffffu, done)) break;
        h = max(h, vF);
        vMaxCol = max(vMaxCol, h);
        Hst[j * 32] = (uint8_t)h;
        vF = max(vF - ge, 0);
        if (++j >= W) {
          j = 0;
          vF = __shfl_up_sync(0xffffffffu, vF, 1);
          if (lane == 0) vF = 0;
        }
      }
      vmax = max(vmax, vMaxCol);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if (lane == 0) P.scores[it] = vmax;
    __syncwarp();
  }
}


// ---------------------------------------------------------------------------------------------
// Stage-1 selection of Prefilter::prefilter_db on the device (src/hhprefilter.cpp:477-506): the N raw scores
// never travel to the host.  Pass 1 applies the length correction (:477) and histograms the corrected scores;
// the host picks the cut from the 1024-bin histogram; pass 2 compacts the survivors.
// ---------------------------------------------------------------------------------------------
constexpr int kPfHistBins = 1024;   // bin = corrected score + 512, clamped
constexpr int kPfHistBias = 512;

__global__ void __launch_bounds__(256)
k_pf_correct_hist(int n, const int* __restrict__ L, const int* __restrict__ raw, float flog2_Lq, int bit_factor,
                  int* __restrict__ corr, unsigned int* __restrict__ hist) {
  __shared__ unsigned int sh[kPfHistBins];
  for (int b = threadIdx.x; b < kPfHistBins; b += blockDim.x) sh[b] = 0;
  __syncthreads();
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const int c = raw[k] - (int)__fmul_rn((float)bit_factor, __fadd_rn(flog2_Lq, flog2_dev((float)L[k])));
    corr[k] = c;
    atomicAdd(&sh[min(max(c + kPfHistBias, 0), kPfHistBins - 1)], 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < kPfHistBins; b += blockDim.x)
    if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// survivors: corr > cut  -> list A;  corr == cut && take_eq -> list B  (order restored by the caller's sort)
__global__ void __launch_bounds__(256)
k_pf_compact(int n, const int* __restrict__ corr, int cut, int take_eq, int* __restrict__ ids_a,
             int* __restrict__ score_a, int* __restrict__ ids_b, unsigned int* __restrict__ counters) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = k < n ? corr[k] : INT_MIN;
  const bool a = k < n && c > cut;
  const bool b = k < n && take_eq && c == cut;
  const unsigned ma = __ballot_sync(0xffffffffu, a), mb = __ballot_sync(0xffffffffu, b);
  const int lane = threadIdx.x & 31;
  unsigned base_a = 0, base_b = 0;
  if (lane == 0) {
    if (ma) base_a = atomicAdd(&counters[0], (unsigned)__popc(ma));
    if (mb) base_b = atomicAdd(&counters[1], (unsigned)__popc(mb));
  }
  base_a = __shfl_sync(0xffffffffu, base_a, 0);
  base_b = __shfl_sync(0xffffffffu, base_b, 0);
  const unsigned below = (1u << lane) - 1u;
  if (a) { const unsigned pos = base_a + __popc(ma & below); ids_a[pos] = k; score_a[pos] = c; }
  if (b) ids_b[base_b + __popc(mb & below)] = k;
}

}  // namespace hhg
