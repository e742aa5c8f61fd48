// General tensor-core path of the recurrent forecaster (LSTM cell, point-estimate head): every shape the H=256 / L=1
// cluster kernels of lstm_tc.cu do not cover -- H a multiple of 64 up to 512, stacked layers, dropout and recurrent
// dropout (BASELINE configs[2]: H=512, L=2, dropout) -- and the fp32-tolerance mode LFMQ_PREC_BF16X3.
//
// One tcgen05 tile-GEMM skeleton (TMA ring -> tcgen05.mma -> TMEM -> epilogue warps) with three epilogues:
//   EPI_FWD    z_t = [h_{t-1} (*rec mask) | in_t] [U; W]   (one launch per time step and layer)
//              epilogue = bias, gate nonlinearities, c_t / h_t update, h_t -> next step's A operand, saved state
//   EPI_BWD    rec = dz_{t+1} U^T                           (one launch per time step and layer, reverse time)
//              epilogue = BPTT pointwise algebra of step t (SURVEY App. A.4) -> dz_t, carried dLoss/dc
//   EPI_STORE  C = A B^T as bf16 (dLoss/d(input) of layers above the first: dz W^T)
// Why launches per time step and not one persistent kernel here: [U; W] of H=512 is 2-4 MB in bf16 -- it fits neither one
// SM nor a portable cluster's shared memory next to the operand ring, so the weight tiles stream from L2 every step
// either way; with two CTAs per SM the epilogue of one tile overlaps the loads / MMAs of the other.  The H=256, L=1 case
// (weights resident in a 4-CTA cluster for the whole unroll) keeps its persistent kernels in lstm_tc.cu.
//
// Data layout (time-major, Bp = maxB rounded up to 128 rows, "blocked" = [..][row tile][16-unit block][piece][4 warps]
// [32 lanes][16] so that a warp's 32-byte-per-thread access is 1 KB contiguous):
//   hseq[l]  bf16 [T+1][Bp][H]    slot t = h_{t-1} (slot 0 zero): A operand of step t, input of BN/Dropout, A^T of dU
//   hmseq[l] bf16 [T+1][Bp][H]    recurrent dropout only: h_{t-1} * mask (what the recurrence and dU actually consume)
//   in[l]    bf16 [T][Bp][Ipad]   layer input (l = 0: x cast to bf16; l > 0: Dropout(BN(h_{l-1}))); in[L] feeds the head
//   gates[l] bf16 blocked [T][row tile][H/16][4 gates]   post-activation i, f, g, o;  cst[l] blocked [T][row tile][H/16]
//   dz       bf16 [T][Bp][4H]     gate pre-activation gradients, standard column order i|f|g|o (shared by the layers)
//   dy / dhout bf16 [T][Bp][H]    dLoss/dy_l (from the head or the layer above) and after Dropout/BN backward
#include "rnn_tc.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include <vector>

#include "kernels.h"
#include "sm100.cuh"

namespace lfmq {

using namespace sm100;

namespace {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// bf16 2-D map over a row-major [outer][inner] buffer, SWIZZLE_128B boxes of box_inner (= 64) x box_outer elements.
int gmap_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer) {
  static PFN_encodeTiled enc = nullptr;
  if (!enc) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    LFMQ_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    enc = reinterpret_cast<PFN_encodeTiled>(fn);
    if (!enc) {
      LFMQ_SET_ERR("cuTensorMapEncodeTiled not available");
      return LFMQ_ERR_CUDA;
    }
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    LFMQ_SET_ERR("cuTensorMapEncodeTiled failed with %d (inner %llu outer %llu box %u x %u)", (int)r,
                 (unsigned long long)inner, (unsigned long long)outer, box_inner, box_outer);
    return LFMQ_ERR_CUDA;
  }
  return 0;
}

inline long cdivl(long a, long b) { return (a + b - 1) / b; }

}  // namespace

// =============================================================================================
// Tile GEMM skeleton
// =============================================================================================
// warp 0: TMA producer, warp 1: MMA issuer, then 4 epilogue warps (one TMEM lane quadrant each) per 128-row M tile
constexpr int G_MAXSEG = 6;
constexpr int GBAR_N = 4096;       // step-barrier counters per handle: one per (persistent launch, row-tile group)

// One K segment: n_kb 64-wide k-blocks, A columns from a_col0 of map a_map, B columns from b_col0 of map b_map.
struct GSeg {
  int a_map, b_map, n_kb, a_col0, b_col0;
};
struct GArgs {
  int n_seg;
  GSeg seg[G_MAXSEG];
  int a_row_base;      // A row coordinate = a_row_base + 128 * (MT * blockIdx.x + rt_off)
  int b_row_base;      // B row coordinate = b_row_base + BN * blockIdx.y
  int rt_off;          // first 128-row tile of this launch (the batch can be split over two concurrent launches)
  // Persistent mode (n_steps > 1): one launch runs n_steps consecutive time steps of a layer; step i works on A rows
  // a_row_base + i * row_step with EpiParams::t + i * t_step.  The A operand of a CTA's next step is written by the
  // gridDim.y CTAs of its own row-tile group (same blockIdx.x, all column tiles), so the steps are separated by one
  // barrier PER ROW-TILE GROUP (a counter in global memory; every CTA of the launch resident at once), not by a launch
  // boundary: CTA dispatch, barrier init, TMEM allocation and the wait for the whole previous grid to retire are paid
  // once, and the row-tile groups drift apart instead of hitting HBM in lockstep.
  int n_steps, row_step, t_step;
  int lin_cols;        // > 0: 1-D grid, CTA i = (row tile i / lin_cols, column tile i % lin_cols): the column tiles of a row
                       // tile are dispatched together and share its A tile in L2 (multi-wave GEMMs: EPI_STORE)
  unsigned int* gbar;  // [gridDim.x], zeroed before the launch; counts the group's CTAs that have finished a step
};

enum { EPI_FWD = 0, EPI_BWD = 1, EPI_STORE = 2, EPI_FWD_ACC = 3, EPI_HEAD = 4 };   // _ACC: expf / tanhf (bf16x3)

struct EpiParams {
  // common
  int t, T, B, Bp, H, NRT, NB16;
  int64_t row0;
  // forward
  const float* bias;            // [4H] in the packed column order (sigmoid gates pre-scaled by 1/2 unless accurate)
  float* cstate;                // fp32 blocked [row tile][H/16][4][32][16]: c_{t-1} in, c_t out
  __nv_bfloat16* hseq;          // [T+1][Bp][H]
  __nv_bfloat16* hseq_lo;       // bf16x3: low halves of h
  __nv_bfloat16* hmseq;         // recurrent dropout: masked copy (null otherwise)
  __nv_bfloat16* gates;         // blocked, null: do not save
  __nv_bfloat16* cst;           // blocked, null: do not save
  int accurate;                 // 1: expf / tanhf (bf16x3 mode), 0: tanh.approx
  int use_rec;                  // recurrent dropout active
  DropoutKey rkey;
  // backward
  const __nv_bfloat16* dhout;   // [T][Bp][H]
  float* dcstate;               // fp32 blocked, carried dLoss/dc
  __nv_bfloat16* dz;            // [T][Bp][4H]
  int has_rec;                  // t < T-1: the accumulator holds dz_{t+1} U^T
  // store
  __nv_bfloat16* out;           // [rows][ldc]
  int ldc;
  // head (EPI_HEAD): pred = y Wo + bo, weighted MSE (losses.py:55-135), dLoss/dpred
  const float* hy;              // targets [B][T][O] fp32 or null
  const float* hdenom;          // {B_global, mask_count_global}
  const float* hbo;             // [O]
  float* hpreds;                // [B][T][O] fp32 or null
  __nv_bfloat16* hdpb;          // [T*Bp][64] bf16, cols >= 16 stay zero: dLoss/dpred rows (operand of the dy and dWo GEMMs)
  float* hpartial;              // [GH_PART][gridDim.x]
  float hp1, hp2;
  int hO, htarget, htrain;
  long long* trace;             // debug (LFMQ_TRACE_GEN=1): clock64 stamps of CTA (0,0): start, first stage landed, last MMA
                                // issued, accumulator complete, epilogue done
};

// MT = 128-row M tiles per CTA: 1 (two CTAs per SM overlap one tile's epilogue with the other's loads) or 2 (a 256-row
// CTA tile: each B stage feeds two MMAs, which cuts the L2 -> SM operand traffic per FLOP by a third; the stepped GEMMs
// are bound by exactly that traffic, profiles/r02_summary.md).  The ring takes whatever shared memory one / two resident
// CTAs leave: the loads are latency-bound (~5 K cycles per stage under load), bytes in flight are what buys bandwidth.
template <int BN, int MT, int EPI = 0>
struct GSmem {
  static constexpr int EW = (EPI == 1) ? 2 : 1;   // warps per TMEM lane quadrant and M tile (EPI_BWD)
  static constexpr uint32_t A_BYTES = MT * 128 * 128;     // MT x (128 rows x 64 bf16)
  static constexpr uint32_t B_BYTES = BN * 128;
  static constexpr uint32_t STAGE = A_BYTES + B_BYTES;
  // one launch = one wave for the recurrence steps (<= 148 tiles: one CTA per SM, deep ring); the multi-wave GEMMs keep
  // two CTAs per SM
  static constexpr int CTAS_PER_SM = (MT == 1 && (BN >= 256 || EPI == 2 || EPI == 4)) ? 2 : 1;   // (2 = EPI_STORE, 4 = EPI_HEAD)
  static constexpr int NS = (int)((CTAS_PER_SM == 2 ? 98304u : 196608u) / STAGE);
  static constexpr uint32_t BARS = NS * STAGE;
  static constexpr uint32_t TOTAL = BARS + 256 + 1024;    // + alignment slack
  static constexpr int THREADS = 64 + 128 * MT * EW;      // producer + MMA + 4 * EW epilogue warps per M tile
};

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ void rec_mask16(const DropoutKey& k, int64_t grow, int H, int j0, float m[16]) {
  const uint64_t qb = (uint64_t)grow * (uint64_t)(H / 4) + (uint64_t)(j0 / 4);
#pragma unroll
  for (int i = 0; i < 4; ++i) dropout_quad(k, qb + i, m + 4 * i);
}

__device__ __forceinline__ void unpack16(const uint32_t w[8], float v[16]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    v[2 * e] = bf16_lo(w[e]);
    v[2 * e + 1] = bf16_hi(w[e]);
  }
}
__device__ __forceinline__ void pack16(const float v[16], uint32_t w[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) w[e] = pack_bf16x2(v[2 * e], v[2 * e + 1]);
}

// ---- EPI_FWD: gates, cell update, h_t (SURVEY App. A.1; rnn_point_estimate.py:80-87) ----------------------------
// Accumulator columns of a tile: [16-unit block][gate i|f|g|o][16] (the packed order of the B operand rows).
template <int BN, bool ACC>
__device__ __forceinline__ void epi_fwd(const EpiParams& p, uint32_t tmem, int q, int lane, int rt, const float* bias_s) {
  const int m = q * 32 + lane;
  const long b = (long)rt * 128 + m;
  const bool valid = b < p.B;
  const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
  constexpr int U = BN / 4;                         // hidden units of this tile
  const int unit0 = blockIdx.y * U;
  // c_{t-1} of the NEXT block is kept in flight while the current one is worked on (an L2 round trip per block otherwise)
  float cnext[16];
  const long cs_blk = 4L * 32 * 16;                 // cstate elements per 16-unit block
  float* cs0 = p.cstate + ((((long)rt * p.NB16 + (unit0 >> 4)) * 4 + q) * 32 + lane) * 16;
  if (p.t > 0) {
    ld_global_v8f(cs0, cnext);
    ld_global_v8f(cs0 + 8, cnext + 8);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) cnext[j] = 0.f;
  }
#pragma unroll 1
  for (int blk = 0; blk < U / 16; ++blk) {
    const int j0 = unit0 + blk * 16;
    const int gblk = j0 >> 4;
    uint32_t vi[16], vf[16], vg[16], vo[16];
    const uint32_t ta = tmem + lane_addr + blk * 64;
    tmem_ld_32x32b_x16(ta + 0, vi);
    tmem_ld_32x32b_x16(ta + 16, vf);
    tmem_ld_32x32b_x16(ta + 32, vg);
    tmem_ld_32x32b_x16(ta + 48, vo);
    float cprev[16];
    float* cs = cs0 + blk * cs_blk;
#pragma unroll
    for (int j = 0; j < 16; ++j) cprev[j] = cnext[j];
    if (p.t > 0 && blk + 1 < U / 16) {
      ld_global_v8f(cs + cs_blk, cnext);
      ld_global_v8f(cs + cs_blk + 8, cnext + 8);
    }
    tmem_ld_wait();
    const float* bs = bias_s + blk * 64;          // this tile's packed bias, staged in shared memory (broadcast reads)
    float gi[16], gf[16], gg[16], go[16], cn[16], hv[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float zi = __uint_as_float(vi[j]) + bs[j];
      const float zf = __uint_as_float(vf[j]) + bs[16 + j];
      const float zg = __uint_as_float(vg[j]) + bs[32 + j];
      const float zo = __uint_as_float(vo[j]) + bs[48 + j];
      if (ACC) {
        gi[j] = sigmoid_acc(zi); gf[j] = sigmoid_acc(zf); gg[j] = tanhf(zg); go[j] = sigmoid_acc(zo);
      } else {      // sigmoid(z) = 0.5 tanh(z/2) + 0.5; the 1/2 is folded into the packed weights and bias
        gi[j] = fmaf(0.5f, tanh_approx(zi), 0.5f);
        gf[j] = fmaf(0.5f, tanh_approx(zf), 0.5f);
        gg[j] = tanh_approx(zg);
        go[j] = fmaf(0.5f, tanh_approx(zo), 0.5f);
      }
      cn[j] = fmaf(gf[j], cprev[j], gi[j] * gg[j]);
      hv[j] = go[j] * (ACC ? tanhf(cn[j]) : tanh_approx(cn[j]));
    }
    st_global_v8f(cs, cn);
    st_global_v8f(cs + 8, cn + 8);
    if (valid) {
      const long hoff = ((long)(p.t + 1) * p.Bp + b) * p.H + j0;
      uint32_t w[8];
      pack16(hv, w);
      st_global_v8(p.hseq + hoff, w);
      if (p.hseq_lo) {        // bf16x3: h = hi + lo with |lo| <= 2^-9 |h|
        float lo[16];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          lo[2 * e] = hv[2 * e] - bf16_lo(w[e]);
          lo[2 * e + 1] = hv[2 * e + 1] - bf16_hi(w[e]);
        }
        uint32_t wl[8];
        pack16(lo, wl);
        st_global_v8(p.hseq_lo + hoff, wl);
      }
      if (p.hmseq) {
        float mk[16];
        rec_mask16(p.rkey, p.row0 + b, p.H, j0, mk);
#pragma unroll
        for (int j = 0; j < 16; ++j) mk[j] *= hv[j];
        uint32_t wm[8];
        pack16(mk, wm);
        st_global_v8(p.hmseq + hoff, wm);
      }
      if (p.gates) {
        const long sb = (((long)p.t * p.NRT + rt) * p.NB16 + gblk);
        __nv_bfloat16* gp = p.gates + (((sb * 4 + 0) * 4 + q) * 32 + lane) * 16;
        const long gstride = 4L * 32 * 16;           // between gates
        pack16(gi, w); st_global_v8(gp, w);
        pack16(gf, w); st_global_v8(gp + gstride, w);
        pack16(gg, w); st_global_v8(gp + 2 * gstride, w);
        pack16(go, w); st_global_v8(gp + 3 * gstride, w);
        pack16(cn, w);
        st_global_v8(p.cst + ((sb * 4 + q) * 32 + lane) * 16, w);
      }
    }
  }
}

// ---- EPI_BWD: BPTT pointwise algebra of step t (SURVEY App. A.4) ----------------------------------------------
// Accumulator columns: hidden units unit0 .. unit0+BN-1 in order (rec = dz_{t+1} U^T, before the recurrent mask).
// The saved gates / cell states come from HBM (~1.5 K cycles per dependent load): each warp keeps the operands of its
// NEXT 16-unit block in flight while it works on the current one, and `ew` warps per lane quadrant split the blocks
// (profiles/r02_summary.md: the serial version spent 22 K of a step's 40 K cycles here).
struct BwdOps {
  uint32_t wi[8], wf[8], wg[8], wo[8], wc[8], wcp[8], wd[8];
};

__device__ __forceinline__ void bwd_load_ops(const EpiParams& p, int rt, int q, int lane, long b, bool valid, int j0,
                                             BwdOps& o) {
  if (!valid) {        // rows beyond the batch take part in the warp-collective TMEM loads but touch no memory
#pragma unroll
    for (int e = 0; e < 8; ++e) o.wi[e] = o.wf[e] = o.wg[e] = o.wo[e] = o.wc[e] = o.wcp[e] = o.wd[e] = 0u;
    return;
  }
  const int gblk = j0 >> 4;
  const long gstride = 4L * 32 * 16;
  const long tstride_c = (long)p.NRT * p.NB16 * 4 * 32 * 16;     // cst elements per time step
  const long sb = (((long)p.t * p.NRT + rt) * p.NB16 + gblk);
  const __nv_bfloat16* gp = p.gates + (((sb * 4 + 0) * 4 + q) * 32 + lane) * 16;
  const __nv_bfloat16* cp_ = p.cst + ((sb * 4 + q) * 32 + lane) * 16;
  ld_global_v8(gp, o.wi);
  ld_global_v8(gp + gstride, o.wf);
  ld_global_v8(gp + 2 * gstride, o.wg);
  ld_global_v8(gp + 3 * gstride, o.wo);
  ld_global_v8(cp_, o.wc);
  if (p.t > 0) {
    ld_global_v8(cp_ - tstride_c, o.wcp);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) o.wcp[e] = 0u;
  }
  ld_global_v8(p.dhout + ((long)p.t * p.Bp + b) * p.H + j0, o.wd);
}

// (A prefetch.global.L2 of the next block's operands one block ahead was measured too: 2.635 -> 2.652 ms, dropped.)
__device__ __forceinline__ void bwd_block(const EpiParams& p, uint32_t tmem_blk, int rt, int q, int lane, long b, bool valid,
                                          int j0, const BwdOps& o) {
  const int gblk = j0 >> 4;
  float* dcs = p.dcstate + ((((long)rt * p.NB16 + gblk) * 4 + q) * 32 + lane) * 16;
  float dcc[16];
  if (p.t < p.T - 1 && valid) {
    ld_global_v8f(dcs, dcc);
    ld_global_v8f(dcs + 8, dcc + 8);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) dcc[j] = 0.f;
  }
  float rec[16];
  if (p.has_rec) {
    uint32_t vr[16];
    tmem_ld_32x32b_x16(tmem_blk, vr);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) rec[j] = __uint_as_float(vr[j]);
    if (p.use_rec) {
      float mk[16];
      rec_mask16(p.rkey, p.row0 + b, p.H, j0, mk);
#pragma unroll
      for (int j = 0; j < 16; ++j) rec[j] *= mk[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) rec[j] = 0.f;
  }
  __nv_bfloat16* dzr = p.dz + ((long)p.t * p.Bp + b) * 4 * p.H + j0;
  // Gate-gradient algebra in packed bf16x2 (all operands arrive packed, dz leaves packed; a third of the instructions of
  // the fp32 form, which made this epilogue issue-bound); only the carried dLoss/dc stays in fp32.  SURVEY App. A.4.
  uint32_t zi[8], zf[8], zg[8], zo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {          // two units per packed word
    const uint32_t i2 = o.wi[e], f2 = o.wf[e], g2 = o.wg[e], o2 = o.wo[e];
    const uint32_t dh2 = add_bf16x2(o.wd[e], pack_bf16x2(rec[2 * e], rec[2 * e + 1]));
    const uint32_t tc2 = tanh_bf16x2(o.wc[e]);
    const uint32_t omtc2 = fma_bf16x2(neg_bf16x2(tc2), tc2, BF16X2_ONE);        // 1 - tanh(c)^2
    const uint32_t t1 = mul_bf16x2(mul_bf16x2(dh2, o2), omtc2);                 // dh * o * (1 - tc^2)
    const float dcn0 = dcc[2 * e] + bf16_lo(t1);
    const float dcn1 = dcc[2 * e + 1] + bf16_hi(t1);
    dcc[2 * e] = dcn0 * bf16_lo(f2);
    dcc[2 * e + 1] = dcn1 * bf16_hi(f2);
    const uint32_t dcn2 = pack_bf16x2(dcn0, dcn1);
    const uint32_t omi = fma_bf16x2(neg_bf16x2(i2), i2, i2);                    // i (1 - i)
    const uint32_t omf = fma_bf16x2(neg_bf16x2(f2), f2, f2);                    // f (1 - f)
    const uint32_t omg = fma_bf16x2(neg_bf16x2(g2), g2, BF16X2_ONE);            // 1 - g^2
    const uint32_t omo = fma_bf16x2(neg_bf16x2(o2), o2, o2);                    // o (1 - o)
    zi[e] = mul_bf16x2(dcn2, mul_bf16x2(g2, omi));
    zf[e] = mul_bf16x2(dcn2, mul_bf16x2(o.wcp[e], omf));
    zg[e] = mul_bf16x2(dcn2, mul_bf16x2(i2, omg));
    zo[e] = mul_bf16x2(mul_bf16x2(dh2, tc2), omo);
  }
  if (valid) {
    st_global_v8f(dcs, dcc);
    st_global_v8f(dcs + 8, dcc + 8);
  } else {             // rows beyond the batch: dz exactly zero (the weight-gradient GEMM sums over all rows)
#pragma unroll
    for (int e = 0; e < 8; ++e) zi[e] = zf[e] = zg[e] = zo[e] = 0u;
  }
  // (row-major 32-byte pieces, one line per lane: a store-free timing run put their cost at up to 0.44 ms per train step of
  //  BASELINE configs[2], profiles/r02_summary.md c27; they stay row-major because dz is a TMA-loaded GEMM operand)
  st_global_v8(dzr, zi);
  st_global_v8(dzr + (long)p.H, zf);
  st_global_v8(dzr + 2L * p.H, zg);
  st_global_v8(dzr + 3L * p.H, zo);
}

// `part` of `nparts` warps of this lane quadrant: blocks part, part + nparts, ...
template <int BN>
__device__ __forceinline__ void epi_bwd(const EpiParams& p, uint32_t tmem, int q, int lane, int rt, int part, int nparts) {
  const int m = q * 32 + lane;
  const long b = (long)rt * 128 + m;
  const bool valid = b < p.B;
  const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
  const int unit0 = blockIdx.y * BN;
  constexpr int NB = BN / 16;
  // tcgen05.ld is warp-collective (.sync.aligned): every lane of the warp runs the block loop, also those whose row lies
  // beyond the batch (a ragged last tile) -- they load nothing and store zeros.  (An early return of those lanes hung
  // the kernel, profiles/r02_summary.md.)
  // One block at a time, all of its nine loads issued together.  (Keeping the next block's operands in flight as well
  // needs 2 x 56 registers: at the 168-register cap of a 320-thread CTA that spilled ~100 values per block, and with
  // 198 KB of shared memory in use the L1 that would catch the spills is ~30 KB -- the epilogue took 25 K cycles whatever
  // the arithmetic looked like, profiles/r02_summary.md.)
  BwdOps A;
#pragma unroll 1
  for (int blk = part; blk < NB; blk += nparts) {
    bwd_load_ops(p, rt, q, lane, b, valid, unit0 + blk * 16, A);
    bwd_block(p, tmem + lane_addr + blk * 16, rt, q, lane, b, valid, unit0 + blk * 16, A);
  }
}

// ---- EPI_STORE: accumulator -> bf16 row-major ---------------------------------------------------------------------
template <int BN>
__device__ __forceinline__ void epi_store(const EpiParams& p, uint32_t tmem, int q, int lane, long row, int by) {
  const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
  __nv_bfloat16* o = p.out + row * p.ldc + (long)by * BN;
#pragma unroll 1
  for (int c0 = 0; c0 < BN; c0 += 32) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(tmem + lane_addr + c0, v);
    tmem_ld_wait();
    uint32_t w[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) w[e] = pack_bf16x2(__uint_as_float(v[2 * e]), __uint_as_float(v[2 * e + 1]));
    st_global_v8(o + c0, w);
    st_global_v8(o + c0 + 16, w + 8);
  }
}

// ---- EPI_HEAD: Dense + weighted MSE + dLoss/dpred on the accumulator of pred = y Wo (N = 16) ---------------------------
// One CTA = one 128-row tile (t, rt) of the time-major head input; thread = row.  (rnn_point_estimate.py:105;
// model_utils/losses.py:55-135; SURVEY App. A.3)
constexpr int GH_O = 16;
constexpr int GH_PART = GH_O + 4;      // dbo | s0 s1 s2
__device__ __forceinline__ void epi_head(const EpiParams& p, uint32_t tmem, int q, int lane, float* red_s) {
  const int tile = blockIdx.x;
  const int t = tile / p.NRT, rt = tile % p.NRT;
  const int m = q * 32 + lane;
  const long b = (long)rt * 128 + m;
  const bool valid = b < p.B;
  if (m < GH_PART) red_s[m] = 0.f;
  named_bar_sync(1, 128);
  uint32_t v[16];
  tmem_ld_32x32b_x16(tmem + ((uint32_t)(q * 32) << 16), v);
  const long r = b * p.T + t;          // row of the caller's [B][T][O] tensors
  float yt[GH_O];
#pragma unroll
  for (int k = 0; k < GH_O; ++k) yt[k] = 0.f;
  if (p.hy && valid)
    for (int k = 0; k < p.hO; ++k) yt[k] = p.hy[r * p.hO + k];
  tmem_ld_wait();
  float pr[GH_O];
#pragma unroll
  for (int k = 0; k < GH_O; ++k) pr[k] = (k < p.hO) ? __uint_as_float(v[k]) + __ldg(p.hbo + k) : 0.f;
  if (p.hpreds && valid)
    for (int k = 0; k < p.hO; ++k) p.hpreds[r * p.hO + k] = pr[k];
  if (!p.hy) return;
  float c_all = 0.f, c_last = 0.f, c_tar = 0.f;
  if (p.htrain) {
    const float Bg = p.hdenom[0], Mg = p.hdenom[1];
    c_all = (1.f - p.hp1) * (1.f - p.hp2) / ((float)p.hO * Mg);
    c_last = (1.f - p.hp1) * p.hp2 / (Bg * (float)p.hO);
    c_tar = p.hp1 / Bg;
  }
  bool any = false;
#pragma unroll
  for (int k = 0; k < GH_O; ++k) any |= (yt[k] != 0.0f);          // losses.py:72
  const float mk = (any && valid) ? 1.f : 0.f;
  const bool last = (t == p.T - 1);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f;
  float dp[GH_O];
#pragma unroll
  for (int k = 0; k < GH_O; ++k) {
    const float d = (k < p.hO && valid) ? (pr[k] * mk - yt[k]) : 0.f;  // losses.py:75
    const float d2 = d * d;
    s2 += d2;
    float coef = c_all;
    if (last) {
      s1 += d2;
      coef += c_last;
      if (k == p.htarget) {
        s0 += d2;
        coef += c_tar;
      }
    }
    dp[k] = p.htrain ? 2.f * d * coef * mk : 0.f;
  }
  if (p.htrain) {       // every row of the tile is written (zeros beyond the batch): the dy / dWo GEMMs run over all rows
    uint32_t w[8];
    pack16(dp, w);
    st_global_v8(p.hdpb + ((long)t * p.Bp + b) * 64, w);
  }
  s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
#pragma unroll
  for (int k = 0; k < GH_O; ++k) dp[k] = warp_sum(dp[k]);
  if (lane == 0) {
    atomicAdd(&red_s[GH_O + 0], s0);
    atomicAdd(&red_s[GH_O + 1], s1);
    atomicAdd(&red_s[GH_O + 2], s2);
    if (p.htrain)
      for (int k = 0; k < GH_O; ++k) atomicAdd(&red_s[k], dp[k]);
  }
  named_bar_sync(1, 128);
  if (m < GH_PART) p.hpartial[(long)m * gridDim.x + blockIdx.x] = red_s[m];
}

template <int BN, int EPI, int MT>
__global__ void __launch_bounds__(GSmem<BN, MT, EPI>::THREADS, GSmem<BN, MT, EPI>::CTAS_PER_SM)
    tile_gemm_kernel(GArgs g, EpiParams ep, const __grid_constant__ CUtensorMap tmA0,
                     const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                     const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmB0,
                     const __grid_constant__ CUtensorMap tmB1) {
  using S = GSmem<BN, MT, EPI>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::BARS);
  uint64_t* empty = full + S::NS;
  uint64_t* acc_full = empty + S::NS;
  uint64_t* tmem_free = acc_full + 1;               // persistent mode: the epilogue has drained the accumulator
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(tmem_free + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr uint32_t TMEM_COLS = (BN * MT < 32) ? 32 : BN * MT;
  __shared__ float red_s[EPI == EPI_HEAD ? GH_PART : 1];
  __shared__ float bias_s[(EPI == EPI_FWD || EPI == EPI_FWD_ACC) ? BN : 1];
  if constexpr (EPI == EPI_FWD || EPI == EPI_FWD_ACC)
    for (int i = tid; i < BN; i += S::THREADS) bias_s[i] = ep.bias[blockIdx.y * BN + i];    // weights: not the predecessor's

  int total_kb = 0;
  for (int i = 0; i < g.n_seg; ++i) total_kb += g.seg[i].n_kb;

  if (tid == 0) {
    for (int s = 0; s < S::NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(tmem_free, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_base_s, TMEM_COLS);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_base_s;
  const int bx = g.lin_cols > 0 ? (int)blockIdx.x / g.lin_cols : (int)blockIdx.x;      // row-tile / column-tile coordinates
  const int by = g.lin_cols > 0 ? (int)blockIdx.x % g.lin_cols : (int)blockIdx.y;
  const bool tr = ep.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0;
  if (tr && tid == 0) ep.trace[0] = clock64();

  // Programmatic dependent launch (the recurrence steps are launched with the stream-serialization attribute): this
  // kernel's CTAs are dispatched while the previous step's grid drains.  Everything above (barriers, TMEM) and the B
  // operand (weights: packed long before the previous step) of the first ring stages is independent of it; the A
  // operand and every state the epilogue reads were written by the previous step, so all threads wait here first.
  // launch_dependents comes AFTER the wait: when the next grid starts, this one has seen its predecessor complete, so
  // by induction only the immediate predecessor can still be running.
  const int n_steps = g.n_steps > 1 ? g.n_steps : 1;
  const unsigned int n_cta = gridDim.y;             // CTAs of this row-tile group
  if (warp == 0) {
    if (lane == 0) {
      const int brow = g.b_row_base + BN * by;
      for (int it = 0; it < n_steps; ++it) {
        const int arow = g.a_row_base + it * g.row_step + 128 * (MT * bx + g.rt_off);
        const int gi0 = it * total_kb;               // ring position of this step's first k-block
        {   // B operand (weights) of the first NS stages of the step, before the dependency wait
          int i = 0;
          for (int sg = 0; sg < g.n_seg && i < S::NS; ++sg) {
            const GSeg sgm = g.seg[sg];
            const CUtensorMap* mb = sgm.b_map == 0 ? &tmB0 : &tmB1;
            for (int kb = 0; kb < sgm.n_kb && i < S::NS; ++kb, ++i) {
              const int gi = gi0 + i, st_ = gi % S::NS;
              if (gi >= S::NS) mbar_wait(&empty[st_], ((gi / S::NS) - 1) & 1);
              mbar_arrive_expect_tx(&full[st_], S::STAGE);
              tma_load_2d(smem + st_ * S::STAGE + S::A_BYTES, mb, &full[st_], sgm.b_col0 + kb * 64, brow);
            }
          }
        }
        long long* trc = tr ? ep.trace + (long)it * g.t_step * 8 : nullptr;     // trace entries are [t][8]
        if (trc && it > 0) trc[0] = clock64();
        if (it == 0) {
          griddep_wait();
          griddep_launch_dependents();
          if (trc) trc[1] = clock64();
        } else {
          // every CTA of the row-tile group has published step it-1 (generic-proxy stores, fenced before the count went up)
          const long long spin0 = clock64();
          while (ld_acquire_gpu(g.gbar + blockIdx.x) < (unsigned int)it * n_cta) {
            // the host only takes this mode when all CTAs fit on the machine at once; should a peer never arrive
            // (SMs held by somebody else), fail the launch after ~2 s instead of hanging the device
            if (clock64() - spin0 > 4000000000LL) __trap();
          }
          fence_proxy_async_global();
          if (trc) trc[1] = clock64();
        }
        int i = 0;
        for (int sg = 0; sg < g.n_seg; ++sg) {
          const GSeg sgm = g.seg[sg];
          const CUtensorMap* ma = sgm.a_map == 0 ? &tmA0 : (sgm.a_map == 1 ? &tmA1 : (sgm.a_map == 2 ? &tmA2 : &tmA3));
          const CUtensorMap* mb = sgm.b_map == 0 ? &tmB0 : &tmB1;
          for (int kb = 0; kb < sgm.n_kb; ++kb, ++i) {
            const int gi = gi0 + i, s = gi % S::NS;
            uint8_t* st = smem + s * S::STAGE;
            if (i >= S::NS) {
              mbar_wait(&empty[s], ((gi / S::NS) - 1) & 1);
              mbar_arrive_expect_tx(&full[s], S::STAGE);
              tma_load_2d(st + S::A_BYTES, mb, &full[s], sgm.b_col0 + kb * 64, brow);
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
              tma_load_2d(st + mt * 16384, ma, &full[s], sgm.a_col0 + kb * 64, arow + 128 * mt);
          }
        }
      }
    } else {
      griddep_wait();
      griddep_launch_dependents();
    }
  } else if (warp == 1) {
    griddep_wait();
    griddep_launch_dependents();
    if (lane == 0 && total_kb > 0) {
      const uint32_t idesc = make_idesc_bf16(128, BN, false, false);
      for (int it = 0; it < n_steps; ++it) {
        if (it > 0) {                          // the epilogue of the previous step has read the accumulator
          mbar_wait(tmem_free, (it - 1) & 1);
          tcgen05_fence_after();
        }
        for (int i = 0; i < total_kb; ++i) {
          const int gi = it * total_kb + i, s = gi % S::NS;
          mbar_wait(&full[s], (gi / S::NS) & 1);
          if (tr && i == 0) ep.trace[(long)it * g.t_step * 8 + 2] = clock64();
          tcgen05_fence_after();
          uint8_t* st = smem + s * S::STAGE;
#pragma unroll
          for (int k16 = 0; k16 < 4; ++k16) {
            const uint64_t db = make_smem_desc(smem_u32(st + S::A_BYTES) + k16 * 32, 0, 1024, LAYOUT_SW128);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
              const uint64_t da = make_smem_desc(smem_u32(st + mt * 16384) + k16 * 32, 0, 1024, LAYOUT_SW128);
              umma_f16(tmem + mt * BN, da, db, idesc, (i | k16) != 0);
            }
          }
          umma_commit(&empty[s]);
        }
        umma_commit(acc_full);
        if (tr) ep.trace[(long)it * g.t_step * 8 + 3] = clock64();
      }
    }
  } else {
    griddep_wait();
    griddep_launch_dependents();
    const int q = warp & 3;
    const int grp = (warp - 2) >> 2;                 // group of four warps = one pass over the four TMEM lane quadrants
    const int mt = grp / S::EW;                      // which 128-row M tile of the CTA this group works on
    const int part = grp % S::EW;                    // ... and which share of its column blocks
    const int rt = MT * bx + mt + g.rt_off;        // 128-row tile index
    // (An L2 prefetch of the epilogue's saved-state operands issued here, during the mainloop, was measured and lost:
    //  it delays the operand ring -- first stage 1.5 K -> 3 K cycles -- and the epilogue, which is issue-bound, not
    //  HBM-bound, got no shorter: 2.97 -> 3.25 ms for the backward steps of BASELINE configs[2].)
    const uint32_t tacc = tmem + mt * BN;
    const int t_first = ep.t;
    for (int it = 0; it < n_steps; ++it) {
      ep.t = t_first + it * g.t_step;
      if (total_kb > 0) {
        mbar_wait(acc_full, it & 1);
        tcgen05_fence_after();
      }
      if (tr && warp == 2 && lane == 0) ep.trace[(long)it * g.t_step * 8 + 4] = clock64();
      if constexpr (EPI == EPI_HEAD) {
        epi_head(ep, tacc, q, lane, red_s);
      } else if ((long)rt * 128 < ep.Bp || EPI == EPI_STORE) {      // (a 256-row CTA tile may hang over the last row tile)
        if constexpr (EPI == EPI_FWD) epi_fwd<BN, false>(ep, tacc, q, lane, rt, bias_s);
        if constexpr (EPI == EPI_FWD_ACC) epi_fwd<BN, true>(ep, tacc, q, lane, rt, bias_s);
        if constexpr (EPI == EPI_BWD) epi_bwd<BN>(ep, tacc, q, lane, rt, part, S::EW);
        if constexpr (EPI == EPI_STORE) epi_store<BN>(ep, tacc, q, lane, (long)g.a_row_base + 128L * rt + q * 32 + lane, by);
      }
      if (tr && warp == 2 && lane == 0) ep.trace[(long)it * g.t_step * 8 + 5] = clock64();
      if (n_steps > 1) {
        // end of a step: all epilogue warps of the CTA are done with the accumulator and have issued their stores; one
        // thread makes them visible device-wide and counts the CTA in (the pattern of a cooperative grid sync)
        tcgen05_fence_before();
        named_bar_sync(2, S::THREADS - 64);
        if (warp == 2 && lane == 0) {
          mbar_arrive(tmem_free);
          __threadfence();
          atomicAdd(g.gbar + blockIdx.x, 1u);
        }
      }
    }
    (void)part;
  }
  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, TMEM_COLS);
}

// =============================================================================================
// Weight gradients: D[M x N] = A^T B over the T*Bp time-major rows, both operands MN-major straight from their
// row-major buffers (the scheme of wgrad_tc_kernel in lstm_tc.cu, for any M, N).  grid = (M tiles of 128, N tiles of
// 256, K splits); deterministic split-K through fp32 partials.
// =============================================================================================
struct GWgradParams {
  int n_kblocks, kb_per_split, Mpad, Ntot;
  float* partial;       // [S][Mpad][Ntot]
};
// MT = 128-row M tiles per CTA (2: a 256 x 256 CTA tile, each B stage feeds two MMAs -- a third less operand traffic
// per FLOP, see GSmem)
template <int MT>
struct GWCfg {
  static constexpr int THREADS = 64 + 128 * MT;
  static constexpr uint32_t A_BYTES = MT * 16384;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + 32768;
  static constexpr int STAGES = (int)(196608u / STAGE_BYTES);       // 4 (MT = 1) or 3 (MT = 2)
  static constexpr uint32_t SMEM = STAGES * STAGE_BYTES + 1024 + 256;
};

template <int MT>
__global__ void __launch_bounds__(GWCfg<MT>::THREADS, 1)
    gwgrad_kernel(GWgradParams p, const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b) {
  using C = GWCfg<MT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty = full + C::STAGES;
  uint64_t* acc_full = empty + C::STAGES;
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * 128 * MT, n0 = blockIdx.y * 256;
  const int kb_beg = blockIdx.z * p.kb_per_split;
  const int kb_end = min(p.n_kblocks, kb_beg + p.kb_per_split);
  const int nkb = max(0, kb_end - kb_beg);
  if (tid == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_base_s, 256 * MT);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_base_s;
  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % C::STAGES;
        if (i >= C::STAGES) mbar_wait(&empty[s], ((i / C::STAGES) - 1) & 1);
        mbar_arrive_expect_tx(&full[s], C::STAGE_BYTES);
        uint8_t* st = smem + s * C::STAGE_BYTES;
        const int krow = (kb_beg + i) * 64;
        for (int mb = 0; mb < 2 * MT; ++mb) tma_load_2d(st + mb * 8192, &tm_a, &full[s], m0 + mb * 64, krow);
        for (int nb = 0; nb < 4; ++nb) tma_load_2d(st + C::A_BYTES + nb * 8192, &tm_b, &full[s], n0 + nb * 64, krow);
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {
      const uint32_t idesc = make_idesc_bf16(128, 256, true, true);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % C::STAGES;
        mbar_wait(&full[s], (i / C::STAGES) & 1);
        tcgen05_fence_after();
        uint8_t* st = smem + s * C::STAGE_BYTES;
#pragma unroll
        for (int k16 = 0; k16 < 4; ++k16) {
          const uint64_t db = make_smem_desc(smem_u32(st + C::A_BYTES) + k16 * 2048, 8192, 1024, LAYOUT_SW128);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            const uint64_t da = make_smem_desc(smem_u32(st + mt * 16384) + k16 * 2048, 8192, 1024, LAYOUT_SW128);
            umma_f16(tmem + mt * 256, da, db, idesc, (i | k16) != 0);
          }
        }
        umma_commit(&empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    const int q = warp & 3;
    const int mt = (warp - 2) >> 2;
    const int m = mt * 128 + q * 32 + lane;
    float* out = p.partial + ((long)blockIdx.z * p.Mpad + m0 + m) * p.Ntot + n0;
    if (nkb > 0) {
      mbar_wait(acc_full, 0);
      tcgen05_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < 256; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem + ((uint32_t)(q * 32) << 16) + mt * 256 + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(out + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                 __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
      }
    } else {
      for (int c0 = 0; c0 < 256; c0 += 4) *reinterpret_cast<float4*>(out + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 256 * MT);
}

// dst[row][n] = sum_z partial[z][row][n] for row < Mvalid (dst row-major [Mvalid][Ntot])
// (rows row_first .. row_first + Mvalid - 1 of the partials)
__global__ void gwgrad_reduce_kernel(int S, int Mvalid, int Mpad, int Ntot, const float* __restrict__ partial,
                                     float* __restrict__ dst, int row_first) {
  const long idx = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (idx >= (long)Mvalid * Ntot) return;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int z = 0; z < S; ++z) {
    const float4 v = *reinterpret_cast<const float4*>(partial + (long)z * Mpad * Ntot + (long)row_first * Ntot + idx);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  *reinterpret_cast<float4*>(dst + idx) = s;
}

// =============================================================================================
// Small streaming kernels
// =============================================================================================
// x f32 [B][T][F] -> in0 bf16 [T][Bp][Ipad] (+ low halves for bf16x3); 8 columns per thread, padding columns zero.
// `ones`: column F (the first padding column) is set to 1 -- the weights of the padding rows are zero, so the forward GEMM
// does not see it, and the weight-gradient GEMM in0^T dz then delivers db = colsum(dz) of the first layer as its row F.
__global__ void gcast_x_kernel(int B, int T, int F, int Bp, int Ipad, const float* __restrict__ x,
                               __nv_bfloat16* __restrict__ o, __nv_bfloat16* __restrict__ o_lo, int ones) {
  const int c8 = Ipad / 8;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)B * T * c8) return;
  const int c = (int)(idx % c8);
  const long r = idx / c8;
  const int t = (int)(r % T);
  const long b = r / T;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int f = c * 8 + e;
    v[e] = (f < F) ? x[(b * T + t) * F + f] : ((ones && f == F) ? 1.f : 0.f);
  }
  uint4 w;
  w.x = pack_bf16x2(v[0], v[1]); w.y = pack_bf16x2(v[2], v[3]); w.z = pack_bf16x2(v[4], v[5]); w.w = pack_bf16x2(v[6], v[7]);
  const long off = ((long)t * Bp + b) * Ipad + c * 8;
  *reinterpret_cast<uint4*>(o + off) = w;
  if (o_lo) {
    uint4 l;
    l.x = pack_bf16x2(v[0] - bf16_lo(w.x), v[1] - bf16_hi(w.x));
    l.y = pack_bf16x2(v[2] - bf16_lo(w.y), v[3] - bf16_hi(w.y));
    l.z = pack_bf16x2(v[4] - bf16_lo(w.z), v[5] - bf16_hi(w.z));
    l.w = pack_bf16x2(v[6] - bf16_lo(w.w), v[7] - bf16_hi(w.w));
    *reinterpret_cast<uint4*>(o_lo + off) = l;
  }
}

// Packed operands of one layer.
//   Wf  [4H][Kp]  forward B operand, K = [h (H) | input (Ipad)], row n = tile*256 + blk*64 + gate*16 + jj  <->  gate column
//                 gate*H + tile*64 + blk*16 + jj of [U; W]; sigmoid gates (i, f, o) pre-scaled by `hs` (0.5, or 1 when accurate)
//   Ub  [H][4H]   backward B operand = recurrent_kernel as it is (rec = dz U^T)
//   Wb  [I][4H]   dLoss/d(input) B operand = kernel as it is (layers above the first)
//   biasp [4H]    bias in Wf's row order, same pre-scale
struct GPackArgs {
  int H, I, Ipad, Kp;
  float hs, eps;
  const float *W, *U, *bias, *gamma, *beta, *mean, *var;
  __nv_bfloat16 *Wf, *Wf_lo, *Ub, *Wb;
  float* biasp;
  float* bn;          // [4][H]: a = gamma * inv | b = beta - mean * a | mean | inv   (BN as the affine map it is here)
};
__global__ void gpack_kernel(GPackArgs a) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int H = a.H;
  const long nWf = (long)4 * H * a.Kp;
  if (idx < nWf) {
    const int k = (int)(idx % a.Kp);
    const int n = (int)(idx / a.Kp);
    const int tile = n / 256, blk = (n % 256) / 64, gate = (n % 64) / 16, jj = n % 16;
    const int col = gate * H + tile * 64 + blk * 16 + jj;
    const float sc = (gate == 2) ? 1.0f : a.hs;
    float v = 0.f;
    if (k < H) v = sc * a.U[(long)k * 4 * H + col];
    else if (k - H < a.I) v = sc * a.W[(long)(k - H) * 4 * H + col];
    const __nv_bfloat16 hi = __float2bfloat16(v);
    a.Wf[idx] = hi;
    if (a.Wf_lo) a.Wf_lo[idx] = __float2bfloat16(v - __bfloat162float(hi));
  }
  if (idx < (long)H * 4 * H && a.Ub) a.Ub[idx] = __float2bfloat16(a.U[idx]);
  if (idx < (long)a.I * 4 * H && a.Wb) a.Wb[idx] = __float2bfloat16(a.W[idx]);
  if (idx < 4 * H) {
    const int n = (int)idx;
    const int tile = n / 256, blk = (n % 256) / 64, gate = (n % 64) / 16, jj = n % 16;
    a.biasp[n] = ((gate == 2) ? 1.0f : a.hs) * a.bias[gate * H + tile * 64 + blk * 16 + jj];
  }
  if (idx < H) {
    const int j = (int)idx;
    const float inv = 1.0f / sqrtf(a.var[j] + a.eps);
    const float ga = a.gamma[j] * inv;
    a.bn[j] = ga;
    a.bn[H + j] = a.beta[j] - a.mean[j] * ga;
    a.bn[2 * H + j] = a.mean[j];
    a.bn[3 * H + j] = inv;
  }
}

// Head operands: WoT [16][H] (B operand of pred = y Wo: row = output k, K = hidden) and WoS [H][64] (B operand of
// dy = dpred Wo^T: row = hidden unit, K = output k, zero beyond O).
__global__ void gpack_head_kernel(int H, int O, const float* __restrict__ Wo, __nv_bfloat16* __restrict__ WoT,
                                  __nv_bfloat16* __restrict__ WoS) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 16 * H) {
    const int k = idx / H, j = idx % H;
    WoT[idx] = __float2bfloat16(k < O ? Wo[j * O + k] : 0.f);
  }
  if (idx < H * 64) {
    const int j = idx / 64, k = idx % 64;
    WoS[idx] = __float2bfloat16(k < O ? Wo[j * O + k] : 0.f);
  }
}

// dWo[j][k] = sum_z partial[z][j][k] (k < O) from the weight-gradient GEMM of the head (N padded to 256)
__global__ void ghead_wo_reduce_kernel(int S, int H, int O, int Mpad, const float* __restrict__ partial,
                                       float* __restrict__ gWo) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= H * O) return;
  const int j = idx / O, k = idx % O;
  float s = 0.f;
  for (int z = 0; z < S; ++z) s += partial[((long)z * Mpad + j) * 256 + k];
  gWo[idx] = s;
}

// y = Dropout(BN(h)) (rnn_point_estimate.py:88-89; BN is the inference affine in both modes, SURVEY App. B #1):
// hseq slots 1..T -> in_next [T][Bp][H] (+ low halves for bf16x3).  8 columns per thread.
__global__ void __launch_bounds__(256)
    gbn_drop_fwd_kernel(int B, int T, int H, int Bp, const __nv_bfloat16* __restrict__ hseq,
                        const __nv_bfloat16* __restrict__ hseq_lo, const float* __restrict__ bn, int use_dropout,
                        DropoutKey key, int64_t row0, __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ y_lo) {
  const int c8 = H / 8;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)T * B * c8) return;
  const int c = (int)(idx % c8);
  const long r = idx / c8;
  const long b = r % B;
  const int t = (int)(r / B);
  const long off = ((long)t * Bp + b) * H + c * 8;
  const uint4 hw = *reinterpret_cast<const uint4*>(hseq + off + (long)Bp * H);      // slot t+1
  float hv[8] = {bf16_lo(hw.x), bf16_hi(hw.x), bf16_lo(hw.y), bf16_hi(hw.y), bf16_lo(hw.z), bf16_hi(hw.z), bf16_lo(hw.w), bf16_hi(hw.w)};
  if (hseq_lo) {
    const uint4 lw = *reinterpret_cast<const uint4*>(hseq_lo + off + (long)Bp * H);
    const float lv[8] = {bf16_lo(lw.x), bf16_hi(lw.x), bf16_lo(lw.y), bf16_hi(lw.y), bf16_lo(lw.z), bf16_hi(lw.z), bf16_lo(lw.w), bf16_hi(lw.w)};
#pragma unroll
    for (int e = 0; e < 8; ++e) hv[e] += lv[e];
  }
  float mk[8];
  if (use_dropout) {
    const uint64_t qb = ((uint64_t)(row0 + b) * T + t) * (uint64_t)(H / 4) + c * 2;
    dropout_quad(key, qb, mk);
    dropout_quad(key, qb + 1, mk + 4);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) mk[e] = 1.f;
  }
  const float4 a0 = __ldg(reinterpret_cast<const float4*>(bn + c * 8)), a1 = __ldg(reinterpret_cast<const float4*>(bn + c * 8 + 4));
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(bn + H + c * 8)), b1 = __ldg(reinterpret_cast<const float4*>(bn + H + c * 8 + 4));
  const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
  const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
  float o[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) o[e] = fmaf(av[e], hv[e], bv[e]) * mk[e];
  uint4 w;
  w.x = pack_bf16x2(o[0], o[1]); w.y = pack_bf16x2(o[2], o[3]); w.z = pack_bf16x2(o[4], o[5]); w.w = pack_bf16x2(o[6], o[7]);
  *reinterpret_cast<uint4*>(y + off) = w;
  if (y_lo) {
    uint4 l;
    l.x = pack_bf16x2(o[0] - bf16_lo(w.x), o[1] - bf16_hi(w.x));
    l.y = pack_bf16x2(o[2] - bf16_lo(w.y), o[3] - bf16_hi(w.y));
    l.z = pack_bf16x2(o[4] - bf16_lo(w.z), o[5] - bf16_hi(w.z));
    l.w = pack_bf16x2(o[6] - bf16_lo(w.w), o[7] - bf16_hi(w.w));
    *reinterpret_cast<uint4*>(y_lo + off) = l;
  }
}

// Dropout / BN backward: dhout = dy * mask * gamma * inv; per-CTA partial sums of dgamma, dbeta (SURVEY App. A.4).
// Thread = 8 columns; a CTA of 256 threads holds 256 / (H/8) rows at a time and walks its row range.
constexpr int GBN_ROWS = 64;
__global__ void __launch_bounds__(256)
    gbn_drop_bwd_kernel(int B, int T, int H, int Bp, const __nv_bfloat16* __restrict__ dy,
                        const __nv_bfloat16* __restrict__ hseq, const float* __restrict__ bn, int use_dropout,
                        DropoutKey key, int64_t row0, __nv_bfloat16* __restrict__ dhout, float* __restrict__ partial) {
  extern __shared__ float red[];      // [RL][2H]
  const int c8 = H / 8;
  const int RL = blockDim.x / c8;
  const int c = threadIdx.x % c8, rl = threadIdx.x / c8;
  float g[8], mu[8], inv[8], sg[8], sb[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int j = c * 8 + e;
    g[e] = bn[j];
    mu[e] = bn[2 * H + j];
    inv[e] = bn[3 * H + j];
    sg[e] = 0.f;
    sb[e] = 0.f;
  }
  const long rows = (long)T * B;
  const long r0 = (long)blockIdx.x * GBN_ROWS;
  const long r1 = min(rows, r0 + GBN_ROWS);
  if (rl < RL) {
#pragma unroll 2
    for (long r = r0 + rl; r < r1; r += RL) {
      const long b = r % B;
      const int t = (int)(r / B);
      const long off = ((long)t * Bp + b) * H + c * 8;
      const uint4 dw = *reinterpret_cast<const uint4*>(dy + off);
      const uint4 hw = *reinterpret_cast<const uint4*>(hseq + off + (long)Bp * H);
      float d[8] = {bf16_lo(dw.x), bf16_hi(dw.x), bf16_lo(dw.y), bf16_hi(dw.y), bf16_lo(dw.z), bf16_hi(dw.z), bf16_lo(dw.w), bf16_hi(dw.w)};
      const float hv[8] = {bf16_lo(hw.x), bf16_hi(hw.x), bf16_lo(hw.y), bf16_hi(hw.y), bf16_lo(hw.z), bf16_hi(hw.z), bf16_lo(hw.w), bf16_hi(hw.w)};
      if (use_dropout) {
        float mk[8];
        const uint64_t qb = ((uint64_t)(row0 + b) * T + t) * (uint64_t)(H / 4) + c * 2;
        dropout_quad(key, qb, mk);
        dropout_quad(key, qb + 1, mk + 4);
#pragma unroll
        for (int e = 0; e < 8; ++e) d[e] *= mk[e];
      }
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        sg[e] += d[e] * (hv[e] - mu[e]) * inv[e];
        sb[e] += d[e];
        o[e] = d[e] * g[e];
      }
      uint4 w;
      w.x = pack_bf16x2(o[0], o[1]); w.y = pack_bf16x2(o[2], o[3]); w.z = pack_bf16x2(o[4], o[5]); w.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(dhout + off) = w;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      red[(long)rl * 2 * H + c * 8 + e] = sg[e];
      red[(long)rl * 2 * H + H + c * 8 + e] = sb[e];
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 2 * H; k += blockDim.x) {
    float sum = 0.f;
    for (int r = 0; r < RL; ++r) sum += red[(long)r * 2 * H + k];
    partial[(long)k * gridDim.x + blockIdx.x] = sum;        // [value][cta]
  }
}

// out[k] = sum over CTAs of partial[k][cta] (one warp per value, fixed order -> deterministic); values [0,n0) go to
// dst0, [n0, n0+n1) to dst1
__global__ void gpartial_reduce_kernel(int n_cta, int n0, int n1, const float* __restrict__ partial,
                                       float* __restrict__ dst0, float* __restrict__ dst1) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= n0 + n1) return;
  double s = 0.0;
  for (int c = lane; c < n_cta; c += 32) s += partial[(long)k * n_cta + c];
  s = warp_sum(s);
  if (lane == 0) {
    if (k < n0) dst0[k] = (float)s;
    else dst1[k - n0] = (float)s;
  }
}

// db = column sums of dz (bf16 [rows][N]) -> partial[column][chunk]; thread = 8 columns (128-bit loads), 4 rows in flight
__global__ void __launch_bounds__(128) gcolsum_kernel(long rows, int N, long rows_per_chunk,
                                                     const __nv_bfloat16* __restrict__ A, float* __restrict__ partial) {
  const int c8 = blockIdx.x * 128 + threadIdx.x;       // group of 8 columns
  if (c8 * 8 >= N) return;
  const long r0 = (long)blockIdx.y * rows_per_chunk, r1 = min(rows, r0 + rows_per_chunk);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  long r = r0;
  for (; r + 4 <= r1; r += 4) {
    uint4 w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const uint4*>(A + (r + u) * N + c8 * 8);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      s[0] += bf16_lo(w[u].x); s[1] += bf16_hi(w[u].x); s[2] += bf16_lo(w[u].y); s[3] += bf16_hi(w[u].y);
      s[4] += bf16_lo(w[u].z); s[5] += bf16_hi(w[u].z); s[6] += bf16_lo(w[u].w); s[7] += bf16_hi(w[u].w);
    }
  }
  for (; r < r1; ++r) {
    const uint4 w = *reinterpret_cast<const uint4*>(A + r * N + c8 * 8);
    s[0] += bf16_lo(w.x); s[1] += bf16_hi(w.x); s[2] += bf16_lo(w.y); s[3] += bf16_hi(w.y);
    s[4] += bf16_lo(w.z); s[5] += bf16_hi(w.z); s[6] += bf16_lo(w.w); s[7] += bf16_hi(w.w);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) partial[(long)(c8 * 8 + e) * gridDim.y + blockIdx.y] = s[e];
}

// =============================================================================================
// Head on y = in[L] (bf16 [T][Bp][H], BN / Dropout already applied): Dense -> weighted MSE -> dpred, dy, loss sums.
// One thread per row of a 128-row tile (TMA-staged, SW128), Wo broadcast from shared memory.
// (rnn_point_estimate.py:105; model_utils/losses.py:55-135; SURVEY App. A.2-A.4)
// =============================================================================================
struct GHeadParams {
  int B, T, O, H, Bp, NRT, target_idx, train;
  const float *Wo, *bo;
  const float* y;            // targets [B][T][O] fp32 (null: predict)
  const float* denom;
  float p1, p2;
  float* preds;              // [B][T][O] fp32 or null
  const __nv_bfloat16* yin_lo;   // bf16x3: low halves of the head input (row-major, same layout), else null
  __nv_bfloat16* dy;         // [T][Bp][H] (train)
  float* dpred;              // [T*Bp][16] fp32 (train)
  float* partial;            // [GH_PART][grid]
};
template <bool TRAIN>
__global__ void __launch_bounds__(128, 1) ghead_rows_kernel(GHeadParams p, const __grid_constant__ CUtensorMap tm_y) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int nkb = p.H / 64;
  float* Wo_s = reinterpret_cast<float*>(tile + (size_t)nkb * 16384);          // [H][16]
  uint64_t* bar = reinterpret_cast<uint64_t*>(Wo_s + (size_t)p.H * GH_O);
  __shared__ float red_s[GH_PART];
  const int tid = threadIdx.x, lane = tid & 31;
  for (int i = tid; i < p.H * GH_O; i += 128) {
    const int j = i / GH_O, k = i % GH_O;
    Wo_s[i] = (k < p.O) ? p.Wo[j * p.O + k] : 0.f;
  }
  for (int i = tid; i < GH_PART; i += 128) red_s[i] = 0.f;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  float c_all = 0.f, c_last = 0.f, c_tar = 0.f;
  if (TRAIN) {
    const float Bg = p.denom[0], Mg = p.denom[1];
    c_all = (1.f - p.p1) * (1.f - p.p2) / ((float)p.O * Mg);
    c_last = (1.f - p.p1) * p.p2 / (Bg * (float)p.O);
    c_tar = p.p1 / Bg;
  }
  float s0 = 0.f, s1 = 0.f, s2 = 0.f;
  float accbo[GH_O];
#pragma unroll
  for (int k = 0; k < GH_O; ++k) accbo[k] = 0.f;
  const int sw = tid & 7;
  uint32_t phase = 0;
  const int n_tiles = p.T * p.NRT;
  for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
    const int t = ti / p.NRT, rt = ti % p.NRT;
    const long b = (long)rt * 128 + tid;
    const bool valid = b < p.B;
    if (tid == 0) {
      mbar_arrive_expect_tx(bar, (uint32_t)nkb * 16384u);
      for (int kb = 0; kb < nkb; ++kb) tma_load_2d(tile + kb * 16384, &tm_y, bar, kb * 64, t * p.Bp + rt * 128);
    }
    const long r = b * p.T + t;          // row of the caller's [B][T][O] tensors
    float yt[GH_O];
#pragma unroll
    for (int k = 0; k < GH_O; ++k) yt[k] = 0.f;
    if (p.y && valid)
      for (int k = 0; k < p.O; ++k) yt[k] = p.y[r * p.O + k];
    mbar_wait(bar, phase);
    phase ^= 1;
    const uint8_t* hrow = tile + tid * 128;
    const __nv_bfloat16* lorow = p.yin_lo ? p.yin_lo + ((long)t * p.Bp + b) * p.H : nullptr;
    float pr[GH_O];
#pragma unroll
    for (int k = 0; k < GH_O; ++k) pr[k] = (k < p.O) ? p.bo[k] : 0.f;
#pragma unroll 2
    for (int c = 0; c < p.H / 8; ++c) {
      const uint4 raw = *reinterpret_cast<const uint4*>(hrow + (c >> 3) * 16384 + (((c & 7) ^ sw) << 4));
      const uint32_t hw[4] = {raw.x, raw.y, raw.z, raw.w};
      uint32_t lw[4] = {0u, 0u, 0u, 0u};
      if (lorow && valid) {
        const uint4 l = *reinterpret_cast<const uint4*>(lorow + c * 8);
        lw[0] = l.x; lw[1] = l.y; lw[2] = l.z; lw[3] = l.w;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int j = c * 8 + e;
        const float yv = ((e & 1) ? bf16_hi(hw[e >> 1]) : bf16_lo(hw[e >> 1])) +
                         ((e & 1) ? bf16_hi(lw[e >> 1]) : bf16_lo(lw[e >> 1]));
        const float4* w4 = reinterpret_cast<const float4*>(Wo_s + j * GH_O);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 w = w4[kk];
          pr[4 * kk + 0] = fmaf(yv, w.x, pr[4 * kk + 0]);
          pr[4 * kk + 1] = fmaf(yv, w.y, pr[4 * kk + 1]);
          pr[4 * kk + 2] = fmaf(yv, w.z, pr[4 * kk + 2]);
          pr[4 * kk + 3] = fmaf(yv, w.w, pr[4 * kk + 3]);
        }
      }
    }
    if (p.preds && valid)
      for (int k = 0; k < p.O; ++k) p.preds[r * p.O + k] = pr[k];
    if (p.y) {
      bool any = false;
#pragma unroll
      for (int k = 0; k < GH_O; ++k) any |= (yt[k] != 0.0f);          // losses.py:72
      const float mk = (any && valid) ? 1.f : 0.f;
      const bool last = (t == p.T - 1);
      float dp[GH_O];
#pragma unroll
      for (int k = 0; k < GH_O; ++k) {
        const float d = (k < p.O && valid) ? (pr[k] * mk - yt[k]) : 0.f;  // losses.py:75
        const float d2 = d * d;
        s2 += d2;
        float coef = c_all;
        if (last) {
          s1 += d2;
          coef += c_last;
          if (k == p.target_idx) {
            s0 += d2;
            coef += c_tar;
          }
        }
        dp[k] = TRAIN ? 2.f * d * coef * mk : 0.f;
        if (TRAIN) accbo[k] += dp[k];
      }
      if (TRAIN) {
        const long rr = (long)t * p.Bp + b;       // time-major row (all 128 rows of the tile are written)
#pragma unroll
        for (int k4 = 0; k4 < GH_O; k4 += 4)
          *reinterpret_cast<float4*>(p.dpred + rr * GH_O + k4) = make_float4(dp[k4], dp[k4 + 1], dp[k4 + 2], dp[k4 + 3]);
        __nv_bfloat16* dyr = p.dy + rr * p.H;
#pragma unroll 1
        for (int c = 0; c < p.H / 16; ++c) {
          float dv[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float4* w4 = reinterpret_cast<const float4*>(Wo_s + (c * 16 + e) * GH_O);
            float sacc = 0.f;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              const float4 w = w4[kk];
              sacc = fmaf(dp[4 * kk + 0], w.x, sacc);
              sacc = fmaf(dp[4 * kk + 1], w.y, sacc);
              sacc = fmaf(dp[4 * kk + 2], w.z, sacc);
              sacc = fmaf(dp[4 * kk + 3], w.w, sacc);
            }
            dv[e] = sacc;
          }
          uint32_t w[8];
          pack16(dv, w);
          st_global_v8(dyr + c * 16, w);
        }
      }
    }
    __syncthreads();        // everyone is done with the tile before it is overwritten
  }
  if (p.y) {
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
#pragma unroll
    for (int k = 0; k < GH_O; ++k) accbo[k] = warp_sum(accbo[k]);
    if (lane == 0) {
      atomicAdd(&red_s[GH_O + 0], s0);
      atomicAdd(&red_s[GH_O + 1], s1);
      atomicAdd(&red_s[GH_O + 2], s2);
      if (TRAIN)
        for (int k = 0; k < GH_O; ++k) atomicAdd(&red_s[k], accbo[k]);
    }
    __syncthreads();
    for (int i = tid; i < GH_PART; i += 128) p.partial[(long)i * gridDim.x + blockIdx.x] = red_s[i];
  }
}

// dWo[j][k] = sum_rows y[row][j] dpred[row][k]: grid (row chunks, H/64); 256 threads = 64 units x 4 groups of 4 outputs.
constexpr int GHW_ROWS = 32;
__global__ void __launch_bounds__(256) ghead_wgrad_kernel(long rows, int H, const __nv_bfloat16* __restrict__ yin,
                                                         const float* __restrict__ dpred, float* __restrict__ wpartial) {
  __shared__ __align__(16) float y_s[GHW_ROWS][64];
  __shared__ __align__(16) float dp_s[GHW_ROWS][GH_O];
  const int tid = threadIdx.x;
  const int j0 = blockIdx.y * 64;
  const int jl = tid >> 2, kg = tid & 3;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (long r0 = (long)blockIdx.x * GHW_ROWS; r0 < rows; r0 += (long)gridDim.x * GHW_ROWS) {
    {   // 32 rows x 64 units = 256 chunks of 8
      const int rr = tid >> 3, ch = tid & 7;
      const long r = r0 + rr;
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (r < rows) {
        const uint4 raw = *reinterpret_cast<const uint4*>(yin + r * H + j0 + ch * 8);
        v[0] = bf16_lo(raw.x); v[1] = bf16_hi(raw.x); v[2] = bf16_lo(raw.y); v[3] = bf16_hi(raw.y);
        v[4] = bf16_lo(raw.z); v[5] = bf16_hi(raw.z); v[6] = bf16_lo(raw.w); v[7] = bf16_hi(raw.w);
      }
      *reinterpret_cast<float4*>(&y_s[rr][ch * 8]) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(&y_s[rr][ch * 8 + 4]) = make_float4(v[4], v[5], v[6], v[7]);
    }
    for (int idx = tid; idx < GHW_ROWS * GH_O; idx += 256) {
      const long r = r0 + idx / GH_O;
      dp_s[idx / GH_O][idx % GH_O] = (r < rows) ? dpred[r * GH_O + idx % GH_O] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < GHW_ROWS; ++rr) {
      const float yv = y_s[rr][jl];
      const float4 dv = *reinterpret_cast<const float4*>(&dp_s[rr][kg * 4]);
      acc[0] = fmaf(yv, dv.x, acc[0]);
      acc[1] = fmaf(yv, dv.y, acc[1]);
      acc[2] = fmaf(yv, dv.z, acc[2]);
      acc[3] = fmaf(yv, dv.w, acc[3]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    wpartial[((long)(j0 + jl) * GH_O + kg * 4 + i) * gridDim.x + blockIdx.x] = acc[i];     // [value][cta]
}

// Sums the head partials: loss terms -> {loss, mse_0}, dbo, dWo.
__global__ void ghead_reduce_kernel(int n_cta, const float* __restrict__ partial, int n_wcta,
                                    const float* __restrict__ wpartial, int H, int O, const float* denom, float p1,
                                    float p2, int train, float* __restrict__ gWo, float* __restrict__ gbo,
                                    float* __restrict__ out2) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;     // one warp per output value
  const int lane = threadIdx.x & 31;
  const int nW = H * GH_O;
  if (i < nW) {
    if (!train || !gWo) return;
    const int j = i / GH_O, k = i % GH_O;
    double s = 0.0;
    for (int c = lane; c < n_wcta; c += 32) s += wpartial[(long)i * n_wcta + c];
    s = warp_sum(s);
    if (lane == 0 && k < O && gWo) gWo[j * O + k] = (float)s;
    return;
  }
  const int q = i - nW;
  if (q >= GH_PART) return;
  double s = 0.0;
  for (int c = lane; c < n_cta; c += 32) s += partial[(long)q * n_cta + c];
  s = warp_sum(s);
  if (q < GH_O) {
    if (train && lane == 0 && q < O) gbo[q] = (float)s;
  } else if (q == GH_O) {
    double s1 = 0.0, s2 = 0.0;
    for (int c = lane; c < n_cta; c += 32) {
      s1 += partial[(long)(q + 1) * n_cta + c];
      s2 += partial[(long)(q + 2) * n_cta + c];
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0 && out2) {
      const double Bg = denom[0], Mg = denom[1];
      const double mse0 = s / Bg, mse1 = s1 / (Bg * O), mse2 = s2 / (Mg * O);
      out2[0] = (float)(p1 * mse0 + (1.0 - p1) * (p2 * mse1 + (1.0 - p2) * mse2));
      out2[1] = (float)mse0;
    }
  }
}

// =============================================================================================
// Host side
// =============================================================================================
struct GenLayer {
  GenLayerOff off;
  int I, Ipad, Kp;
  __nv_bfloat16 *hseq, *hseq_lo, *hmseq, *in, *in_lo, *gates, *cst;
  __nv_bfloat16 *Wf, *Wf_lo, *Ub, *Wb;
  float *biasp, *bn;
  CUtensorMap tm_h, tm_h_lo, tm_hm, tm_in, tm_in_lo, tm_wf, tm_wf_lo, tm_ub, tm_wb;    // K-major (recurrence, dx)
  CUtensorMap tm_hA_mn, tm_in_mn;                                                       // MN-major (weight gradients)
};

struct GenImpl {
  bool enabled = false;
  unsigned int* gbar = nullptr;         // grid-barrier counters of the persistent step launches (GBAR_N, zeroed per call)
  int gbar_next = 0;
  int n_sms = 0;
  cudaStream_t side = nullptr;          // second half of the batch in the backward recurrence (see gen_backward)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  long long* trace = nullptr;      // LFMQ_TRACE_GEN=1: [phase 0 fwd / 1 bwd][layer][t][8] clock64 stamps of CTA (0,0)
  int maxB = 0, Bp = 0, NRT = 0, T = 0, F = 0, O = 0, H = 0, L = 0, NB16 = 0;
  bool x3 = false, train_ws = false;
  int64_t oWo = 0, obo = 0;
  std::vector<GenLayer> layers;
  __nv_bfloat16 *head_in = nullptr, *head_in_lo = nullptr;      // in[L]
  CUtensorMap tm_head_in;
  // tensor-core head (bf16): packed Wo, bf16 dLoss/dpred rows, per-tile loss partials
  __nv_bfloat16 *WoT = nullptr, *WoS = nullptr, *dpb = nullptr;
  float* head_tc_part = nullptr;
  CUtensorMap tm_wot, tm_wos, tm_dpb, tm_dpb_mn, tm_head_in_mn;
  float *cstate = nullptr, *dcstate = nullptr;
  __nv_bfloat16 *dz = nullptr, *dy = nullptr, *dhout = nullptr;
  CUtensorMap tm_dz, tm_dz_mn;
  float *dpred = nullptr, *head_part = nullptr, *head_wpart = nullptr, *bn_part = nullptr, *cs_part = nullptr;
  float* wg_part = nullptr;
  size_t wg_part_elems = 0;
  int head_ctas = 0, head_wctas = 0, bn_ctas_max = 0, cs_chunks = 0;
  int BNU = 128;      // hidden units per backward tile
};

bool gen_supported(const lfmq_config& c, char* why, size_t n) {
  if (c.rnn_cell != LFMQ_CELL_LSTM) { snprintf(why, n, "the tensor-core paths are built for the LSTM cell only"); return false; }
  if (c.uq) { snprintf(why, n, "the tensor-core paths are built for the point-estimate head only"); return false; }
  if (c.num_hidden % 64 != 0 || c.num_hidden > 512) {
    snprintf(why, n, "num_hidden must be a multiple of 64 and <= 512 (got %d)", c.num_hidden);
    return false;
  }
  if (c.n_outputs > GH_O) { snprintf(why, n, "n_outputs must be <= 16 (got %d)", c.n_outputs); return false; }
  if (c.n_inputs > 1024) { snprintf(why, n, "n_inputs must be <= 1024 (got %d)", c.n_inputs); return false; }
  if (c.precision == LFMQ_PREC_BF16X3 && !c.forward_only) {
    snprintf(why, n, "LFMQ_PREC_BF16X3 (fp32-tolerance forward) is built for forward_only handles");
    return false;
  }
  return true;
}

void gen_layout(GenState& st, const lfmq_config& c, const GenLayerOff* lo, int64_t oWo, int64_t obo, char* base,
                size_t& off) {
  if (!st.impl) st.impl = new GenImpl;
  GenImpl& m = *st.impl;
  auto take = [&](size_t bytes) -> char* {
    char* p = base ? base + off : nullptr;
    off = (off + bytes + 1023) / 1024 * 1024;
    return p;
  };
  m.maxB = c.max_batch; m.T = c.seq_len; m.F = c.n_inputs; m.O = c.n_outputs; m.H = c.num_hidden; m.L = c.num_layers;
  m.Bp = (c.max_batch + 127) / 128 * 128;
  m.NRT = m.Bp / 128;
  m.NB16 = m.H / 16;
  m.x3 = c.precision == LFMQ_PREC_BF16X3;
  m.train_ws = !c.forward_only;
  m.oWo = oWo; m.obo = obo;
  m.BNU = (m.H % 128 == 0) ? 128 : 64;   // 64-unit tiles at H % 128 == 0 were slower (profiles/r02_summary.md, c28)
  const size_t T = m.T, Bp = m.Bp, H = m.H;
  const bool rec = (c.train && c.recurrent_dropout > 0.f);
  m.layers.assign(m.L, GenLayer{});
  for (int l = 0; l < m.L; ++l) {
    GenLayer& ly = m.layers[l];
    ly.off = lo[l];
    ly.I = lo[l].I;
    ly.Ipad = (ly.I + 63) / 64 * 64;
    ly.Kp = (int)H + ly.Ipad;
    ly.hseq = reinterpret_cast<__nv_bfloat16*>(take((T + 1) * Bp * H * 2));
    ly.hseq_lo = m.x3 ? reinterpret_cast<__nv_bfloat16*>(take((T + 1) * Bp * H * 2)) : nullptr;
    ly.hmseq = rec ? reinterpret_cast<__nv_bfloat16*>(take((T + 1) * Bp * H * 2)) : nullptr;
    ly.in = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * ly.Ipad * 2));
    ly.in_lo = m.x3 ? reinterpret_cast<__nv_bfloat16*>(take(T * Bp * ly.Ipad * 2)) : nullptr;
    ly.Wf = reinterpret_cast<__nv_bfloat16*>(take((size_t)4 * H * ly.Kp * 2));
    ly.Wf_lo = m.x3 ? reinterpret_cast<__nv_bfloat16*>(take((size_t)4 * H * ly.Kp * 2)) : nullptr;
    ly.biasp = reinterpret_cast<float*>(take(4 * H * 4));
    ly.bn = reinterpret_cast<float*>(take(4 * H * 4));
    if (m.train_ws) {
      ly.gates = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * 4 * H * 2));
      ly.cst = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * H * 2));
      ly.Ub = reinterpret_cast<__nv_bfloat16*>(take(H * 4 * H * 2));
      ly.Wb = (l > 0) ? reinterpret_cast<__nv_bfloat16*>(take((size_t)ly.I * 4 * H * 2)) : nullptr;
    } else {
      ly.gates = ly.cst = ly.Ub = ly.Wb = nullptr;
    }
  }
  m.head_in = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * H * 2));
  m.head_in_lo = m.x3 ? reinterpret_cast<__nv_bfloat16*>(take(T * Bp * H * 2)) : nullptr;
  m.WoT = reinterpret_cast<__nv_bfloat16*>(take(16 * H * 2));
  m.WoS = reinterpret_cast<__nv_bfloat16*>(take(H * 64 * 2));
  m.head_tc_part = reinterpret_cast<float*>(take((size_t)GH_PART * T * m.NRT * 4));
  m.dpb = m.train_ws ? reinterpret_cast<__nv_bfloat16*>(take(T * Bp * 64 * 2)) : nullptr;
  m.cstate = reinterpret_cast<float*>(take(Bp * H * 4));
  m.head_ctas = 148;
  m.head_part = reinterpret_cast<float*>(take((size_t)GH_PART * m.head_ctas * 4));
  if (m.train_ws) {
    m.dcstate = reinterpret_cast<float*>(take(Bp * H * 4));
    m.dz = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * 4 * H * 2));
    m.dy = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * H * 2));
    m.dhout = reinterpret_cast<__nv_bfloat16*>(take(T * Bp * H * 2));
    m.dpred = reinterpret_cast<float*>(take(T * Bp * GH_O * 4));
    m.head_wctas = 148;
    m.head_wpart = reinterpret_cast<float*>(take((size_t)H * GH_O * m.head_wctas * 4));
    m.bn_ctas_max = (int)cdivl((long)T * m.maxB, GBN_ROWS);
    m.bn_part = reinterpret_cast<float*>(take((size_t)2 * H * m.bn_ctas_max * 4));
    m.cs_chunks = 1024;
    m.cs_part = reinterpret_cast<float*>(take((size_t)4 * H * m.cs_chunks * 4));
    const size_t Mmax = (H > 64 ? H : 128);               // dU: H rows; dW: Ipad rows (<= max(H, 64..1024))
    size_t mp = (Mmax + 255) / 256 * 256;
    for (int l = 0; l < m.L; ++l) {
      const size_t ip = ((size_t)m.layers[l].Ipad + 255) / 256 * 256;
      if (ip > mp) mp = ip;
    }
    m.wg_part_elems = (size_t)8 * mp * 4 * H;             // up to 8 K-splits
    m.wg_part = reinterpret_cast<float*>(take(m.wg_part_elems * 4));
  }
}

int gen_init(GenState& st, const lfmq_config& c) {
  char why[160];
  if (!gen_supported(c, why, sizeof(why))) {
    LFMQ_SET_ERR("tensor-core precision unsupported for this configuration: %s; use LFMQ_PREC_FP32", why);
    return LFMQ_ERR_UNSUPPORTED;
  }
  GenImpl& m = *st.impl;
  const size_t T = m.T, Bp = m.Bp, H = m.H;
  int rc;
  for (int l = 0; l < m.L; ++l) {
    GenLayer& ly = m.layers[l];
    // every buffer that is an operand of a GEMM over padded rows / columns must hold finite values everywhere
    LFMQ_CUDA_CHECK(cudaMemset(ly.hseq, 0, (T + 1) * Bp * H * 2));
    if (ly.hseq_lo) LFMQ_CUDA_CHECK(cudaMemset(ly.hseq_lo, 0, (T + 1) * Bp * H * 2));
    if (ly.hmseq) LFMQ_CUDA_CHECK(cudaMemset(ly.hmseq, 0, (T + 1) * Bp * H * 2));
    LFMQ_CUDA_CHECK(cudaMemset(ly.in, 0, T * Bp * ly.Ipad * 2));
    if (ly.in_lo) LFMQ_CUDA_CHECK(cudaMemset(ly.in_lo, 0, T * Bp * ly.Ipad * 2));
    const uint64_t hrows = (T + 1) * Bp;
    if ((rc = gmap_2d(&ly.tm_h, ly.hseq, H, hrows, 64, 128))) return rc;
    if (ly.hseq_lo && (rc = gmap_2d(&ly.tm_h_lo, ly.hseq_lo, H, hrows, 64, 128))) return rc;
    if (ly.hmseq && (rc = gmap_2d(&ly.tm_hm, ly.hmseq, H, hrows, 64, 128))) return rc;
    if ((rc = gmap_2d(&ly.tm_in, ly.in, ly.Ipad, T * Bp, 64, 128))) return rc;
    if (ly.in_lo && (rc = gmap_2d(&ly.tm_in_lo, ly.in_lo, ly.Ipad, T * Bp, 64, 128))) return rc;
    if ((rc = gmap_2d(&ly.tm_wf, ly.Wf, ly.Kp, 4 * H, 64, 256))) return rc;
    if (ly.Wf_lo && (rc = gmap_2d(&ly.tm_wf_lo, ly.Wf_lo, ly.Kp, 4 * H, 64, 256))) return rc;
    if (m.train_ws) {
      if ((rc = gmap_2d(&ly.tm_ub, ly.Ub, 4 * H, H, 64, m.BNU))) return rc;
      if (ly.Wb && (rc = gmap_2d(&ly.tm_wb, ly.Wb, 4 * H, ly.I, 64, (H % 128 == 0) ? 128 : 64))) return rc;
      // MN-major views for the weight gradients: slots 0..T-1 of (hmseq | hseq) against dz, boxes 64 (M) x 64 (rows)
      if ((rc = gmap_2d(&ly.tm_hA_mn, ly.hmseq ? ly.hmseq : ly.hseq, H, T * Bp, 64, 64))) return rc;
      if ((rc = gmap_2d(&ly.tm_in_mn, ly.in, ly.Ipad, T * Bp, 64, 64))) return rc;
    }
  }
  LFMQ_CUDA_CHECK(cudaMemset(m.head_in, 0, T * Bp * H * 2));
  if (m.head_in_lo) LFMQ_CUDA_CHECK(cudaMemset(m.head_in_lo, 0, T * Bp * H * 2));
  if ((rc = gmap_2d(&m.tm_head_in, m.head_in, H, T * Bp, 64, 128))) return rc;
  if ((rc = gmap_2d(&m.tm_wot, m.WoT, H, 16, 64, 16))) return rc;
  if (m.train_ws) {
    LFMQ_CUDA_CHECK(cudaMemset(m.dpb, 0, T * Bp * 64 * 2));       // columns >= 16 stay zero for good
    if ((rc = gmap_2d(&m.tm_wos, m.WoS, 64, H, 64, (H % 128 == 0) ? 128 : 64))) return rc;
    if ((rc = gmap_2d(&m.tm_dpb, m.dpb, 64, T * Bp, 64, 128))) return rc;
    if ((rc = gmap_2d(&m.tm_dpb_mn, m.dpb, 64, T * Bp, 64, 64))) return rc;
    if ((rc = gmap_2d(&m.tm_head_in_mn, m.head_in, H, T * Bp, 64, 64))) return rc;
  }
  if (m.train_ws) {
    LFMQ_CUDA_CHECK(cudaMemset(m.dz, 0, T * Bp * 4 * H * 2));
    LFMQ_CUDA_CHECK(cudaMemset(m.dy, 0, T * Bp * H * 2));
    LFMQ_CUDA_CHECK(cudaMemset(m.dhout, 0, T * Bp * H * 2));
    LFMQ_CUDA_CHECK(cudaMemset(m.dpred, 0, T * Bp * GH_O * 4));
    if ((rc = gmap_2d(&m.tm_dz, m.dz, 4 * H, T * Bp, 64, 128))) return rc;
    if ((rc = gmap_2d(&m.tm_dz_mn, m.dz, 4 * H, T * Bp, 64, 64))) return rc;
  }
#define LFMQ_GEMM_ATTR(BN_, EPI_, MT_)                                                                         \
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(tile_gemm_kernel<BN_, EPI_, MT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                       GSmem<BN_, MT_, EPI_>::TOTAL))
  LFMQ_GEMM_ATTR(256, EPI_FWD, 1);
  LFMQ_GEMM_ATTR(256, EPI_FWD, 2);
  LFMQ_GEMM_ATTR(256, EPI_FWD_ACC, 1);
  LFMQ_GEMM_ATTR(256, EPI_FWD_ACC, 2);
  LFMQ_GEMM_ATTR(128, EPI_BWD, 1);
  LFMQ_GEMM_ATTR(64, EPI_BWD, 1);
  LFMQ_GEMM_ATTR(16, EPI_HEAD, 1);
  LFMQ_GEMM_ATTR(128, EPI_STORE, 1);
  LFMQ_GEMM_ATTR(64, EPI_STORE, 1);
#undef LFMQ_GEMM_ATTR
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(gwgrad_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GWCfg<1>::SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(gwgrad_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GWCfg<2>::SMEM));
  const int hsmem = (int)((H / 64) * 16384 + H * GH_O * 4 + 64 + 1024);
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(ghead_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, hsmem));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(ghead_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, hsmem));
  if (m.train_ws) {
    const int bsm = (256 / ((int)H / 8) > 0 ? 256 / ((int)H / 8) : 1) * 2 * (int)H * 4;
    LFMQ_CUDA_CHECK(cudaFuncSetAttribute(gbn_drop_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bsm));
  }
  if (getenv("LFMQ_TRACE_GEN")) {
    LFMQ_CUDA_CHECK(cudaMalloc(&m.trace, (size_t)2 * m.L * T * 8 * sizeof(long long)));
    LFMQ_CUDA_CHECK(cudaMemset(m.trace, 0, (size_t)2 * m.L * T * 8 * sizeof(long long)));
  }
  LFMQ_CUDA_CHECK(cudaMalloc(&m.gbar, GBAR_N * sizeof(unsigned int)));
  LFMQ_CUDA_CHECK(cudaMemset(m.gbar, 0, GBAR_N * sizeof(unsigned int)));
  {
    int dev = 0;
    LFMQ_CUDA_CHECK(cudaGetDevice(&dev));
    LFMQ_CUDA_CHECK(cudaDeviceGetAttribute(&m.n_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  m.enabled = true;
  st.weights_dirty = 1;
  return 0;
}

// Persistent step launches need every CTA of the launch(es) running at once (they meet at a grid-wide barrier).
// `n_concurrent` launches of `ctas` CTAs each, `per_sm` resident CTAs of that instantiation per SM.  LFMQ_GEN_PERSIST=0
// turns the mode off (one launch per time step, chained with programmatic dependent launch).
static bool gen_can_persist(const GenImpl& m, long ctas, int n_concurrent, int per_sm, int n_steps) {
  static const bool on = !(getenv("LFMQ_GEN_PERSIST") && atoi(getenv("LFMQ_GEN_PERSIST")) == 0);
  return on && n_steps > 1 && m.gbar != nullptr && ctas * n_concurrent <= (long)m.n_sms * per_sm &&
         m.gbar_next + ctas * n_concurrent <= GBAR_N;
}

static void gen_print_trace(GenImpl& m, cudaStream_t s) {
  if (!m.trace) return;
  const size_t n = (size_t)2 * m.L * m.T * 8;
  std::vector<long long> h(n);
  cudaStreamSynchronize(s);
  cudaMemcpy(h.data(), m.trace, n * sizeof(long long), cudaMemcpyDeviceToHost);
  for (int ph = 0; ph < 2; ++ph)
    for (int l = 0; l < m.L; ++l)
      for (int t = 0; t < m.T; t += 8) {
        const long long* r = h.data() + (((size_t)ph * m.L + l) * m.T + t) * 8;
        if (!r[0]) continue;
        fprintf(stderr, "[gtrace %s l=%d t=%2d] wait-passed %lld first-stage %lld mma-issued %lld acc-full %lld epi-done %lld\n",
                ph ? "bwd" : "fwd", l, t, r[1] - r[0], r[2] - r[0], r[3] - r[0], r[4] - r[0], r[5] - r[0]);
      }
}

void gen_destroy(GenState& st) {
  if (st.impl && st.impl->side) {
    cudaStreamSynchronize(st.impl->side);
    cudaEventDestroy(st.impl->ev_fork);
    cudaEventDestroy(st.impl->ev_join);
    cudaStreamDestroy(st.impl->side);
  }
  if (st.impl && st.impl->trace) cudaFree(st.impl->trace);
  if (st.impl && st.impl->gbar) cudaFree(st.impl->gbar);
  delete st.impl;
  st.impl = nullptr;
}

// Launch of one tile_gemm_kernel instantiation; `pdl`: with the programmatic-stream-serialization attribute (the
// kernel waits for its predecessor itself, see the kernel).  LFMQ_GEN_PDL=0 turns the attribute off.
template <int BN, int EPI, int MT>
static int launch_tile_gemm(dim3 grid, cudaStream_t s, bool pdl, const GArgs& g, const EpiParams& ep, const CUtensorMap& a0,
                            const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& a3, const CUtensorMap& b0,
                            const CUtensorMap& b1) {
  static const bool pdl_on = !(getenv("LFMQ_GEN_PDL") && atoi(getenv("LFMQ_GEN_PDL")) == 0);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(GSmem<BN, MT, EPI>::THREADS);
  cfg.dynamicSmemBytes = GSmem<BN, MT, EPI>::TOTAL;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl && pdl_on) ? 1 : 0;
  LFMQ_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tile_gemm_kernel<BN, EPI, MT>, g, ep, a0, a1, a2, a3, b0, b1));
  g_launches++;
  if (debug_sync_on()) {
    fprintf(stderr, "[lfmq launch] tile_gemm<%d,%d,%d> grid %u x %u t=%d ...", BN, EPI, MT, grid.x, grid.y, ep.t);
    fflush(stderr);
    cudaError_t e = cudaDeviceSynchronize();
    fprintf(stderr, " %s\n", cudaGetErrorString(e));
    fflush(stderr);
  }
  return 0;
}

static DropoutKey gkey(const lfmq_config& c, int stream, int64_t step, float rate) {
  DropoutKey k;
  k.k0 = (uint32_t)(c.seed & 0xffffffffu);
  k.k1 = (uint32_t)(c.seed >> 32);
  k.stream = (uint32_t)stream;
  k.step = (uint32_t)(step & 0xffffffff);
  k.thr = (uint32_t)((double)rate * 16777216.0);
  k.scale = 1.0f / (1.0f - rate);
  return k;
}

static int gen_pack(GenState& st, const float* params, float eps, cudaStream_t s) {
  GenImpl& m = *st.impl;
  if (!st.weights_dirty) return 0;
  for (int l = 0; l < m.L; ++l) {
    GenLayer& ly = m.layers[l];
    GPackArgs a;
    a.H = m.H; a.I = ly.I; a.Ipad = ly.Ipad; a.Kp = ly.Kp;
    a.hs = m.x3 ? 1.0f : 0.5f;
    a.eps = eps;
    a.W = params + ly.off.oW; a.U = params + ly.off.oU; a.bias = params + ly.off.ob;
    a.gamma = params + ly.off.ogamma; a.beta = params + ly.off.obeta; a.mean = params + ly.off.omean; a.var = params + ly.off.ovar;
    a.Wf = ly.Wf; a.Wf_lo = ly.Wf_lo; a.Ub = ly.Ub; a.Wb = ly.Wb; a.biasp = ly.biasp; a.bn = ly.bn;
    const long n = (long)4 * m.H * ly.Kp;
    gpack_kernel<<<(int)cdivl(n, 256), 256, 0, s>>>(a);
    LFMQ_LAUNCH_CHECK();
  }
  gpack_head_kernel<<<(int)cdivl((long)m.H * 64, 256), 256, 0, s>>>(m.H, m.O, params + m.oWo, m.WoT, m.WoS);
  LFMQ_LAUNCH_CHECK();
  st.weights_dirty = 0;
  return 0;
}

// all layers' recurrences + BN/Dropout; leaves in[L] (the head input)
static int gen_run_trunk(GenState& st, const lfmq_config& c, const float* params, const float* x, int B, int64_t row0,
                         int64_t step, bool save, cudaStream_t s) {
  GenImpl& m = *st.impl;
  const int T = m.T, H = m.H, Bp = m.Bp;
  const int nrt = (B + 127) / 128;
  const bool rec = c.train && c.recurrent_dropout > 0.f;
  const bool drop = c.train && c.dropout > 0.f;
  static const char* dual_env = getenv("LFMQ_GEN_DUAL");      // 0 / 1 force, unset: by tile count
  const bool dual = dual_env ? atoi(dual_env) != 0 : ((long)((nrt + 1) / 2) * (4 * H / 256) >= 96);
  LFMQ_CUDA_CHECK(cudaMemsetAsync(m.gbar, 0, GBAR_N * sizeof(unsigned int), s));
  m.gbar_next = 0;
  {
    const GenLayer& l0 = m.layers[0];
    const long n = (long)B * T * (l0.Ipad / 8);
    gcast_x_kernel<<<(int)cdivl(n, 256), 256, 0, s>>>(B, T, m.F, Bp, l0.Ipad, x, l0.in, l0.in_lo,
                                                      (save && !m.x3 && l0.Ipad > m.F) ? 1 : 0);
    LFMQ_LAUNCH_CHECK();
  }
  for (int l = 0; l < m.L; ++l) {
    GenLayer& ly = m.layers[l];
    EpiParams ep = {};
    ep.T = T; ep.B = B; ep.Bp = Bp; ep.H = H; ep.NRT = m.NRT; ep.NB16 = m.NB16; ep.row0 = row0;
    ep.bias = ly.biasp; ep.cstate = m.cstate; ep.hseq = ly.hseq; ep.hseq_lo = ly.hseq_lo;
    ep.hmseq = rec ? ly.hmseq : nullptr;
    ep.gates = save ? ly.gates : nullptr;
    ep.cst = save ? ly.cst : nullptr;
    ep.accurate = m.x3 ? 1 : 0;
    ep.use_rec = rec ? 1 : 0;
    ep.rkey = gkey(c, 2 * l + 1, step, c.recurrent_dropout);
    const CUtensorMap& th = rec ? ly.tm_hm : ly.tm_h;
    // steps 1 .. T-1 as ONE persistent launch when all its CTAs fit on the machine at once (see GArgs::n_steps)
    const long fwd_ctas = dual ? (long)((nrt + 1) / 2) * (4 * H / 256) : (long)nrt * (4 * H / 256);
    const bool persist = gen_can_persist(m, fwd_ctas, 1, dual ? 1 : 2, T - 1);
    for (int t = 0; t < T; ++t) {
      ep.t = t;
      ep.trace = m.trace ? m.trace + (((size_t)0 * m.L + l) * T + t) * 8 : nullptr;
      GArgs g = {};
      g.a_row_base = t * Bp;
      g.b_row_base = 0;
      if (persist && t == 1) {
        g.n_steps = T - 1;
        g.row_step = Bp;
        g.t_step = 1;
        g.gbar = m.gbar + m.gbar_next;
        m.gbar_next += dual ? (nrt + 1) / 2 : nrt;
      }
      const int nkb_h = (t > 0) ? H / 64 : 0, nkb_x = ly.Ipad / 64;
      int ns = 0;
      // maps: A0 = h (or masked h), A1 = input, A2 = h low halves, A3 = input low halves; B0 = weights, B1 = their low halves
      if (nkb_h) g.seg[ns++] = GSeg{0, 0, nkb_h, 0, 0};
      g.seg[ns++] = GSeg{1, 0, nkb_x, 0, H};
      if (m.x3) {
        if (nkb_h) g.seg[ns++] = GSeg{2, 0, nkb_h, 0, 0};      // lo(h) hi(W)
        g.seg[ns++] = GSeg{3, 0, nkb_x, 0, H};
        if (nkb_h) g.seg[ns++] = GSeg{0, 1, nkb_h, 0, 0};      // hi(h) lo(W)
        g.seg[ns++] = GSeg{1, 1, nkb_x, 0, H};
      }
      g.n_seg = ns;
      // 256-row CTA tiles when there are enough of them to fill the machine (a third less operand traffic per FLOP),
      // else 128-row tiles, two CTAs per SM.  Steps after the first of a layer follow another step kernel: PDL.
      int rc;
#define LFMQ_FWD_LAUNCH(EPI_, MT_, GRID_)                                                                          \
  rc = launch_tile_gemm<256, EPI_, MT_>(GRID_, s, t > 0, g, ep, th, ly.tm_in, m.x3 ? ly.tm_h_lo : th,               \
                                        m.x3 ? ly.tm_in_lo : ly.tm_in, ly.tm_wf, m.x3 ? ly.tm_wf_lo : ly.tm_wf)
      const dim3 grid2((nrt + 1) / 2, 4 * H / 256), grid1(nrt, 4 * H / 256);
      if (m.x3) {
        if (dual) LFMQ_FWD_LAUNCH(EPI_FWD_ACC, 2, grid2);
        else LFMQ_FWD_LAUNCH(EPI_FWD_ACC, 1, grid1);
      } else {
        if (dual) LFMQ_FWD_LAUNCH(EPI_FWD, 2, grid2);
        else LFMQ_FWD_LAUNCH(EPI_FWD, 1, grid1);
      }
#undef LFMQ_FWD_LAUNCH
      if (rc) return rc;
      if (persist && t == 1) break;              // that launch ran steps 1 .. T-1
    }
    const bool last = (l == m.L - 1);
    __nv_bfloat16* yo = last ? m.head_in : m.layers[l + 1].in;
    __nv_bfloat16* yo_lo = last ? m.head_in_lo : m.layers[l + 1].in_lo;
    const long n = (long)T * B * (H / 8);
    gbn_drop_fwd_kernel<<<(int)cdivl(n, 256), 256, 0, s>>>(B, T, H, Bp, ly.hseq, ly.hseq_lo, ly.bn, drop ? 1 : 0,
                                                           gkey(c, 2 * l, step, c.dropout), row0, yo, yo_lo);
    LFMQ_LAUNCH_CHECK();
  }
  return 0;
}

// D[Mvalid x Ntot] = A^T B over the T*Bp time-major rows (split-K partials in wg_part, [S][Mpad][Ntot]); the caller reduces
static int gen_wgrad_gemm(GenImpl& m, const CUtensorMap& tm_a, const CUtensorMap& tm_b, int Mvalid, int Ntot, int* S_out,
                          int* Mpad_out, cudaStream_t s) {
  const bool dual = Mvalid > 128;                    // 256 x 256 CTA tiles when there are at least two 128-row M tiles
  const int mrows = dual ? 256 : 128;
  const int mt = (Mvalid + mrows - 1) / mrows;
  const int Mpad = mt * mrows;
  const long rows = (long)m.T * m.Bp;
  GWgradParams wp;
  wp.n_kblocks = (int)cdivl(rows, 64);
  // K splits: fill the machine, within what the partial buffer holds (the head's [H x 16] product has one N tile and
  // wants many splits; the gate products have 8-16 output tiles and get 8)
  int S = 148 / (mt * (Ntot / 256));
  const size_t smax = m.wg_part_elems / ((size_t)Mpad * Ntot);
  if ((size_t)S > smax) S = (int)smax;
  if (S > 64) S = 64;
  if (S < 1) S = 1;
  if (S > wp.n_kblocks) S = wp.n_kblocks;
  wp.kb_per_split = (wp.n_kblocks + S - 1) / S;
  S = (wp.n_kblocks + wp.kb_per_split - 1) / wp.kb_per_split;
  wp.Mpad = Mpad;
  wp.Ntot = Ntot;
  wp.partial = m.wg_part;
  if ((size_t)S * Mpad * Ntot > m.wg_part_elems) {
    LFMQ_SET_ERR("weight-gradient partial buffer too small");
    return LFMQ_ERR_WORKSPACE;
  }
  if (dual)
    gwgrad_kernel<2><<<dim3(mt, Ntot / 256, S), GWCfg<2>::THREADS, GWCfg<2>::SMEM, s>>>(wp, tm_a, tm_b);
  else
    gwgrad_kernel<1><<<dim3(mt, Ntot / 256, S), GWCfg<1>::THREADS, GWCfg<1>::SMEM, s>>>(wp, tm_a, tm_b);
  LFMQ_LAUNCH_CHECK();
  *S_out = S;
  *Mpad_out = Mpad;
  return 0;
}

// `db` (nullable): row Mvalid of the product (A's constant-one column, see gcast_x_kernel) = colsum(dz)
static int gen_wgrad(GenImpl& m, const CUtensorMap& tm_a, int Mvalid, float* dst, cudaStream_t s, float* db = nullptr) {
  const int Ntot = 4 * m.H;
  int S = 0, Mpad = 0, rc;
  if ((rc = gen_wgrad_gemm(m, tm_a, m.tm_dz_mn, db ? Mvalid + 1 : Mvalid, Ntot, &S, &Mpad, s))) return rc;
  const long n4 = (long)Mvalid * Ntot / 4;
  gwgrad_reduce_kernel<<<(int)cdivl(n4, 256), 256, 0, s>>>(S, Mvalid, Mpad, Ntot, m.wg_part, dst, 0);
  LFMQ_LAUNCH_CHECK();
  if (db) {
    gwgrad_reduce_kernel<<<(int)cdivl(Ntot / 4, 256), 256, 0, s>>>(S, 1, Mpad, Ntot, m.wg_part, db, Mvalid);
    LFMQ_LAUNCH_CHECK();
  }
  return 0;
}

static int gen_run_head(GenState& st, const lfmq_config& c, const float* params, float* grads, const float* y, int B,
                        const float* denom, float* preds, float* out2, bool train, cudaStream_t s) {
  GenImpl& m = *st.impl;
  GHeadParams h = {};
  h.B = B; h.T = m.T; h.O = m.O; h.H = m.H; h.Bp = m.Bp; h.NRT = (B + 127) / 128; h.target_idx = c.target_idx;
  h.train = train ? 1 : 0;
  h.Wo = params + m.oWo; h.bo = params + m.obo;
  h.y = y; h.denom = denom; h.p1 = c.target_lambda; h.p2 = c.rnn_lambda;
  h.preds = preds;
  h.yin_lo = m.head_in_lo;
  h.dy = train ? m.dy : nullptr;
  h.dpred = train ? m.dpred : nullptr;
  h.partial = m.head_part;
  if (!m.x3) {
    // Tensor-core head: pred = y Wo as a tcgen05 GEMM (N = 16) with the loss in its epilogue; training adds
    // dy = dpred Wo^T (K = 16 padded to one k-block) and dWo = y^T dpred (the weight-gradient GEMM, N padded to 256).
    // The fp32-accumulating SIMT head below stays for LFMQ_PREC_BF16X3 (1e-4 tolerance).
    const int ntile = m.T * m.NRT;                  // every row tile of the time-major buffers (zeros beyond the batch)
    EpiParams ep = {};
    ep.T = m.T; ep.B = B; ep.Bp = m.Bp; ep.H = m.H; ep.NRT = m.NRT; ep.NB16 = m.NB16;
    ep.hy = y; ep.hdenom = denom; ep.hbo = params + m.obo; ep.hpreds = preds; ep.hdpb = m.dpb;
    ep.hpartial = m.head_tc_part; ep.hp1 = c.target_lambda; ep.hp2 = c.rnn_lambda; ep.hO = m.O;
    ep.htarget = c.target_idx; ep.htrain = train ? 1 : 0;
    GArgs g = {};
    g.n_seg = 1;
    g.seg[0] = GSeg{0, 0, m.H / 64, 0, 0};
    int rc;
    if ((rc = launch_tile_gemm<16, EPI_HEAD, 1>(dim3(ntile, 1), s, false, g, ep, m.tm_head_in, m.tm_head_in, m.tm_head_in,
                                                m.tm_head_in, m.tm_wot, m.tm_wot)))
      return rc;
    if (train) {
      EpiParams es = {};
      es.out = m.dy;
      es.ldc = m.H;
      es.Bp = m.Bp;
      GArgs gd = {};
      gd.n_seg = 1;
      gd.seg[0] = GSeg{0, 0, 1, 0, 0};
      const int row_tiles = m.T * m.Bp / 128;
      gd.lin_cols = (m.H % 128 == 0) ? m.H / 128 : m.H / 64;
      if (m.H % 128 == 0)
        rc = launch_tile_gemm<128, EPI_STORE, 1>(dim3(row_tiles * (m.H / 128)), s, false, gd, es, m.tm_dpb, m.tm_dpb, m.tm_dpb,
                                                 m.tm_dpb, m.tm_wos, m.tm_wos);
      else
        rc = launch_tile_gemm<64, EPI_STORE, 1>(dim3(row_tiles * (m.H / 64)), s, false, gd, es, m.tm_dpb, m.tm_dpb, m.tm_dpb,
                                                m.tm_dpb, m.tm_wos, m.tm_wos);
      if (rc) return rc;
      int S = 0, Mpad = 0;
      if ((rc = gen_wgrad_gemm(m, m.tm_head_in_mn, m.tm_dpb_mn, m.H, 256, &S, &Mpad, s))) return rc;
      ghead_wo_reduce_kernel<<<(m.H * m.O + 255) / 256, 256, 0, s>>>(S, m.H, m.O, Mpad, m.wg_part, grads + m.oWo);
      LFMQ_LAUNCH_CHECK();
    }
    if (y) {
      const int n_out = m.H * GH_O + GH_PART;
      ghead_reduce_kernel<<<(n_out * 32 + 255) / 256, 256, 0, s>>>(ntile, m.head_tc_part, 0, nullptr, m.H, m.O, denom,
                                                                 c.target_lambda, c.rnn_lambda, train ? 1 : 0, nullptr,
                                                                 grads ? grads + m.obo : nullptr, out2);
      LFMQ_LAUNCH_CHECK();
    }
    return 0;
  }
  int grid = m.T * h.NRT;
  if (grid > m.head_ctas) grid = m.head_ctas;
  const int hsmem = (m.H / 64) * 16384 + m.H * GH_O * 4 + 64 + 1024;
  if (train)
    ghead_rows_kernel<true><<<grid, 128, hsmem, s>>>(h, m.tm_head_in);
  else
    ghead_rows_kernel<false><<<grid, 128, hsmem, s>>>(h, m.tm_head_in);
  LFMQ_LAUNCH_CHECK();
  int n_wcta = 0;
  if (train) {
    // rows of the time-major buffers: T * Bp (rows >= B of a tile carry dpred = 0)
    const long rows = (long)m.T * m.Bp;
    n_wcta = m.head_wctas;
    ghead_wgrad_kernel<<<dim3(n_wcta, m.H / 64), 256, 0, s>>>(rows, m.H, m.head_in, m.dpred, m.head_wpart);
    LFMQ_LAUNCH_CHECK();
  }
  if (y) {
    const int n_out = m.H * GH_O + GH_PART;
    ghead_reduce_kernel<<<(n_out * 32 + 255) / 256, 256, 0, s>>>(grid, m.head_part, n_wcta, m.head_wpart, m.H, m.O, denom,
                                                               c.target_lambda, c.rnn_lambda, train ? 1 : 0,
                                                               grads ? grads + m.oWo : nullptr,
                                                               grads ? grads + m.obo : nullptr, out2);
    LFMQ_LAUNCH_CHECK();
  }
  return 0;
}

int gen_forward(GenState& st, const lfmq_config& c, const float* params, const float* x, int B, int64_t row0,
                int64_t step, float* preds, cudaStream_t s) {
  if (!st.impl || !st.impl->enabled) {
    LFMQ_SET_ERR("general tensor-core path not initialised");
    return LFMQ_ERR_UNSUPPORTED;
  }
  int rc;
  if ((rc = gen_pack(st, params, c.bn_epsilon, s))) return rc;
  st.prof->begin(LFMQ_REGION_FWD, s);
  if ((rc = gen_run_trunk(st, c, params, x, B, row0, step, false, s))) return rc;
  st.prof->end(LFMQ_REGION_FWD, s);
  st.prof->begin(LFMQ_REGION_HEAD, s);
  if ((rc = gen_run_head(st, c, params, nullptr, nullptr, B, nullptr, preds, nullptr, false, s))) return rc;
  st.prof->end(LFMQ_REGION_HEAD, s);
  return 0;
}

int gen_backward(GenState& st, const lfmq_config& c, const float* params, float* grads, const float* x, const float* y,
                 int B, int64_t row0, int64_t step, const float* denom, float* tail, cudaStream_t s) {
  if (!st.impl || !st.impl->enabled || !st.impl->train_ws) {
    LFMQ_SET_ERR("general tensor-core path not initialised for training");
    return LFMQ_ERR_UNSUPPORTED;
  }
  GenImpl& m = *st.impl;
  const int T = m.T, H = m.H, Bp = m.Bp;
  const int nrt = (B + 127) / 128;
  const bool rec = c.train && c.recurrent_dropout > 0.f;
  const bool drop = c.train && c.dropout > 0.f;
  int rc;
  if ((rc = gen_pack(st, params, c.bn_epsilon, s))) return rc;
  st.prof->begin(LFMQ_REGION_FWD, s);
  if ((rc = gen_run_trunk(st, c, params, x, B, row0, step, true, s))) return rc;
  st.prof->end(LFMQ_REGION_FWD, s);
  if (nrt < m.NRT) {
    // a smaller batch than an earlier call on this handle: the weight-gradient GEMMs sum over all T*Bp time-major rows,
    // so the rows of the row tiles that are not launched now must be zero (they may hold an earlier call's values)
    const size_t tail_rows = (size_t)(Bp - nrt * 128);
    LFMQ_CUDA_CHECK(cudaMemset2DAsync(m.dz + (size_t)nrt * 128 * 4 * H, (size_t)Bp * 4 * H * 2, 0, tail_rows * 4 * H * 2, T, s));
    LFMQ_CUDA_CHECK(cudaMemset2DAsync(m.dpred + (size_t)nrt * 128 * GH_O, (size_t)Bp * GH_O * 4, 0, tail_rows * GH_O * 4, T, s));
  }
  st.prof->begin(LFMQ_REGION_HEAD, s);
  if ((rc = gen_run_head(st, c, params, grads, y, B, denom, nullptr, tail, true, s))) return rc;
  st.prof->end(LFMQ_REGION_HEAD, s);
  for (int l = m.L - 1; l >= 0; --l) {
    GenLayer& ly = m.layers[l];
    st.prof->begin(LFMQ_REGION_BWD, s);
    {   // Dropout / BN backward of this layer's output: dy -> dhout, dgamma, dbeta
      const int ctas = (int)cdivl((long)T * B, GBN_ROWS);
      const int RL = 256 / (H / 8) > 0 ? 256 / (H / 8) : 1;
      gbn_drop_bwd_kernel<<<ctas, 256, RL * 2 * H * 4, s>>>(B, T, H, Bp, m.dy, ly.hseq, ly.bn, drop ? 1 : 0,
                                                           gkey(c, 2 * l, step, c.dropout), row0, m.dhout, m.bn_part);
      LFMQ_LAUNCH_CHECK();
      gpartial_reduce_kernel<<<(2 * H * 32 + 255) / 256, 256, 0, s>>>(ctas, H, H, m.bn_part, grads + ly.off.ogamma,
                                                                    grads + ly.off.obeta);
      LFMQ_LAUNCH_CHECK();
    }
    EpiParams ep = {};
    ep.T = T; ep.B = B; ep.Bp = Bp; ep.H = H; ep.NRT = m.NRT; ep.NB16 = m.NB16; ep.row0 = row0;
    ep.gates = ly.gates; ep.cst = ly.cst; ep.dhout = m.dhout; ep.dcstate = m.dcstate; ep.dz = m.dz;
    ep.use_rec = rec ? 1 : 0;
    ep.rkey = gkey(c, 2 * l + 1, step, c.recurrent_dropout);
    // The step's epilogue is HBM-bound (saved gates / cell states in, dz out: ~46 MB per step at H = 512) and its
    // mainloop L2-bound, and one launch puts every CTA into the same phase at the same time.  Two half-batches on two
    // streams (each its own PDL chain) drift apart, so one half's epilogue runs beside the other's mainloop.
    static const char* split_env = getenv("LFMQ_GEN_SPLIT");      // 0 / 1 force, unset: by tile count
    const bool split = split_env ? (atoi(split_env) != 0 && nrt >= 2) : (nrt >= 16);
    const int n_a = split ? (nrt + 1) / 2 : nrt, n_b = nrt - n_a;
    if (split) {
      if (!m.side) {
        LFMQ_CUDA_CHECK(cudaStreamCreateWithFlags(&m.side, cudaStreamNonBlocking));
        LFMQ_CUDA_CHECK(cudaEventCreateWithFlags(&m.ev_fork, cudaEventDisableTiming));
        LFMQ_CUDA_CHECK(cudaEventCreateWithFlags(&m.ev_join, cudaEventDisableTiming));
      }
      LFMQ_CUDA_CHECK(cudaEventRecord(m.ev_fork, s));
      LFMQ_CUDA_CHECK(cudaStreamWaitEvent(m.side, m.ev_fork, 0));
    }
    // steps T-2 .. 0 of each chain as ONE persistent launch when all CTAs of both chains fit on the machine at once
    const long bwd_ctas = (long)n_a * (H / m.BNU);
    const bool persist = gen_can_persist(m, bwd_ctas, split ? 2 : 1, 1, T - 1);
    for (int t = T - 1; t >= 0; --t) {
      for (int half = 0; half < (split ? 2 : 1); ++half) {       // launches interleaved: neither chain lags the other
        cudaStream_t hs = half ? m.side : s;
        const int rt_off = half ? n_a : 0, n_rt = half ? n_b : n_a;
        ep.t = t;
        ep.trace = (m.trace && half == 0) ? m.trace + (((size_t)1 * m.L + l) * T + t) * 8 : nullptr;
        ep.has_rec = (t < T - 1) ? 1 : 0;
        GArgs g = {};
        g.a_row_base = (t + 1) * Bp;      // dz_{t+1}
        g.b_row_base = 0;
        g.rt_off = rt_off;
        g.n_seg = ep.has_rec ? 1 : 0;
        g.seg[0] = GSeg{0, 0, 4 * H / 64, 0, 0};
        if (persist && t == T - 2) {
          g.n_steps = T - 1;
          g.row_step = -Bp;
          g.t_step = -1;
          g.gbar = m.gbar + m.gbar_next;
          m.gbar_next += n_rt;
        }
        if (m.BNU == 128)
          rc = launch_tile_gemm<128, EPI_BWD, 1>(dim3(n_rt, H / 128), hs, t < T - 1, g, ep, m.tm_dz, m.tm_dz, m.tm_dz,
                                                 m.tm_dz, ly.tm_ub, ly.tm_ub);
        else
          rc = launch_tile_gemm<64, EPI_BWD, 1>(dim3(n_rt, H / 64), hs, t < T - 1, g, ep, m.tm_dz, m.tm_dz, m.tm_dz,
                                                m.tm_dz, ly.tm_ub, ly.tm_ub);
        if (rc) return rc;
      }
      if (persist && t == T - 2) break;          // those launches ran steps T-2 .. 0
    }
    if (split) {
      LFMQ_CUDA_CHECK(cudaEventRecord(m.ev_join, m.side));
      LFMQ_CUDA_CHECK(cudaStreamWaitEvent(s, m.ev_join, 0));
    }
    st.prof->end(LFMQ_REGION_BWD, s);
    st.prof->begin(LFMQ_REGION_WGRAD, s);
    if ((rc = gen_wgrad(m, ly.tm_hA_mn, H, grads + ly.off.oU, s))) return rc;
    // first layer: the input buffer's first padding column is constant one (gcast_x_kernel), so db falls out of the dW GEMM
    const bool ones_db = (l == 0) && !m.x3 && ly.Ipad > ly.I;
    if ((rc = gen_wgrad(m, ly.tm_in_mn, ly.I, grads + ly.off.oW, s, ones_db ? grads + ly.off.ob : nullptr))) return rc;
    if (!ones_db) {   // db = column sums of dz over the T*Bp rows (rows beyond the batch are zero)
      const long rows = (long)T * Bp;
      const long rpc = cdivl(rows, m.cs_chunks);
      gcolsum_kernel<<<dim3((4 * H / 8 + 127) / 128, m.cs_chunks), 128, 0, s>>>(rows, 4 * H, rpc, m.dz, m.cs_part);
      LFMQ_LAUNCH_CHECK();
      gpartial_reduce_kernel<<<(4 * H * 32 + 255) / 256, 256, 0, s>>>(m.cs_chunks, 4 * H, 0, m.cs_part,
                                                                    grads + ly.off.ob, nullptr);
      LFMQ_LAUNCH_CHECK();
    }
    if (l > 0) {   // dLoss/dy_{l-1} = dz W^T  -> dy (bf16 [T*Bp][H])
      EpiParams es = {};
      es.out = m.dy;
      es.ldc = H;
      GArgs g = {};
      g.a_row_base = 0;
      g.b_row_base = 0;
      g.n_seg = 1;
      g.seg[0] = GSeg{0, 0, 4 * H / 64, 0, 0};
      const int row_tiles = T * Bp / 128;
      g.lin_cols = (H % 128 == 0) ? H / 128 : H / 64;
      if (H % 128 == 0)
        rc = launch_tile_gemm<128, EPI_STORE, 1>(dim3(row_tiles * (H / 128)), s, false, g, es, m.tm_dz, m.tm_dz, m.tm_dz,
                                                 m.tm_dz, ly.tm_wb, ly.tm_wb);
      else
        rc = launch_tile_gemm<64, EPI_STORE, 1>(dim3(row_tiles * (H / 64)), s, false, g, es, m.tm_dz, m.tm_dz, m.tm_dz,
                                                m.tm_dz, ly.tm_wb, ly.tm_wb);
      if (rc) return rc;
    }
    st.prof->end(LFMQ_REGION_WGRAD, s);
  }
  (void)x;
  gen_print_trace(m, s);
  return 0;
}

}  // namespace lfmq
