// LFMQ_PREC_BF16: the gate GEMMs on tcgen05 tensor cores (bf16 operands, fp32 accumulation in TMEM, fp32 cell
// state in registers, bf16 when saved), everything else as fused HBM-streaming kernels.  sm_100a only.
//
// Data layout in HBM (all carved from the caller's workspace, see tc_layout):
//   xh    bf16 [maxB][T+1][384]   row (b,t): cols 0..255 = h_{t-1} (zero at t=0), 256..287 = x_t, 288 = 1.0 (t<T),
//                                 rest 0.  One buffer serves: the A operand of the forward recurrence (K-major
//                                 tiles via TMA), the head (h_t = row t+1) and the weight-gradient GEMM (MN-major).
//   gates bf16 [T][tiles][8 blocks of 32 units][4 warps][8 pieces = gate*2+half][32 lanes][16]   post-activation
//                                 i|f|g|o saved for BPTT.  Writer (forward) and reader (backward) both map one
//                                 row to one thread, so the state is stored SoA at 32-byte granularity: a warp's
//                                 256-bit access to `piece` covers 1 KB contiguously instead of 32 scattered sectors
//   cst   bf16 [T][tiles][8][4][2 pieces][32][16]   cell states (the recurrence itself keeps them in fp32 registers)
//   dz    bf16 [maxB][T+1][4H]    gate pre-activation gradients (row T stays zero); columns in the order the
//                                 backward kernel stages them as its A operand, [16-unit block][gate][16], so that a
//                                 chunk goes out with one TMA store; only the weight-gradient GEMM reads it
//   dpb   bf16 [T][tiles][128][32]  dLoss/dpred tiles (cols >= 16 zero): written by the tensor-core head as it stages
//                                 them, expanded to dLoss/dh by the backward kernel's own MMAs (no dropout)
//   dhout bf16 [T][tiles][4 ranks][4 warps][4 chunks][32 lanes][16]   dropout > 0 only: dLoss/dh from the SIMT head
//                                 (after BN/dropout backward), already in the backward kernel's per-thread SoA order
//
// Forward recurrence = ONE persistent kernel (lstm_fwd_tc_kernel): clusters of 4 CTAs, one 128-row batch tile per
// cluster, all clusters co-resident.  CTA r keeps the weight slice of hidden units [64r, 64r+64) (all four gates,
// 256 gate columns) resident in shared memory for the whole unroll.  h_t is exchanged through global memory (it is
// an output anyway) and comes back as the next step's A operand via TMA multicast -- measured on B200
// (profiles/r01_tc_probe.txt) that path moves 64 KB into every SM of a cluster in ~1500 cycles while DSMEM stores
// or bulk copies manage only 9-13 B/cycle/SM.  Clusters of 8 were tried first and dropped: only 15 of them are
// co-resident.  See DESIGN.md section 5 for the per-step cycle budget of both recurrences.
#include "lstm_tc.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "kernels.h"
#include "sm100.cuh"

namespace lfmq {

using namespace sm100;

namespace {

constexpr int TC_H = 256;          // hidden units (bf16 path is specialised for H = 256)
constexpr int TC_NC = 4;           // CTAs per forward cluster
constexpr int TC_HS = 64;          // hidden units per forward CTA
constexpr int TC_NSL = 256;        // gate columns per forward CTA
constexpr int TC_XH_LD = 384;      // elements per xh row
constexpr int TC_XOFF = 256;       // first x column inside an xh row
constexpr int TC_ONE = 288;        // the constant-one column (db falls out of the weight-gradient GEMM)
constexpr int TC_OPAD = 16;        // head handles n_outputs <= 16

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle sw) {
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
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    LFMQ_SET_ERR("cuTensorMapEncodeTiled failed with %d (inner %llu outer %llu box %u x %u)", (int)r,
                 (unsigned long long)inner, (unsigned long long)outer, box_inner, box_outer);
    return LFMQ_ERR_CUDA;
  }
  return 0;
}

// General tiled map (bf16): dims / box innermost first, strides in bytes for dims 1..rank-1.
int make_map_nd(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                const uint32_t* box, CUtensorMapSwizzle sw) {
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
  cuuint64_t d[5], st[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), d, st, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    LFMQ_SET_ERR("cuTensorMapEncodeTiled (rank %d) failed with %d", rank, (int)r);
    return LFMQ_ERR_CUDA;
  }
  return 0;
}

}  // namespace

struct TcImpl {
  bool enabled = false;
  int maxB = 0, T = 0, I = 0, O = 0;
  float eps = 1e-3f;
  // parameter offsets in the flat fp32 vector (L = 1)
  int64_t oW, oU, ob, ogamma, obeta, oWo, obo, omean, ovar;
  // workspace
  __nv_bfloat16 *xh, *gates, *dz, *dhout, *Up, *Wp, *Ubk, *pexch;
  __nv_bfloat16* cst;
  float *biasp, *head_part, *head_wpart, *dpred, *wg_part, *dc;
  size_t head_part_elems, wg_part_elems;
  CUtensorMap tm_h, tm_x, tm_u, tm_w;          // forward
  CUtensorMap tm_h128, tm_wot;                 // head: 128-row h tiles, folded head weights
  __nv_bfloat16* WoTp;
  __nv_bfloat16* WoSp;                         // [256][32]  Wo[j][k] * gamma_j * inv_j (k < 16), zero padded
  __nv_bfloat16* dpb;                          // [T][tiles][128][32] bf16 dLoss/dpred tiles (cols >= 16 zero)
  CUtensorMap tm_wos, tm_dpb;
  float* bop;
  CUtensorMap tm_ubk;                          // backward recurrence
  CUtensorMap tm_xh_mn, tm_dz_mn;              // weight gradient (MN-major)
  int max_clusters = 0, bwd_max_clusters = 0;
  bool bwd_ready = false;
  // L2 prefetch helper for the backward recurrence (LFMQ_BWD_PREFETCH=1): runs on the SMs the recurrence leaves idle
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  unsigned long long* progress = nullptr;      // device: steps completed by the backward kernel, counted across calls
  unsigned long long epoch = 0;
  int head_ctas = 0, head_wctas = 0;
  // head beside the forward recurrence (head_paced_kernel; LFMQ_FWD_HEAD=0 turns it off, read when the handle is made)
  bool fwd_head = false;
  int sm_count = 0;
  unsigned int* head_progress = nullptr;       // device [n_tiles_cap]: forward CTA-steps published per row tile
};

// =============================================================================================
// Small packing / cast kernels
// =============================================================================================
// x f32 [B,T,F] -> xh[b][t][256 .. 256+F), plus the constant-one column.  One 16-byte chunk per thread.
__global__ void xh_fill_x_kernel(int B, int T, int F, const float* __restrict__ x, __nv_bfloat16* __restrict__ xh) {
  pdl_sync();
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;   // (row, chunk) with 5 chunks of 8 columns per row
  if (idx >= (long)B * T * 5) return;
  const long row = idx / 5;
  const int c = (int)(idx % 5);
  const long b = row / T;
  const int t = (int)(row % T);
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int f = c * 8 + e;
    v[e] = (f < F) ? x[row * F + f] : ((f == TC_ONE - TC_XOFF) ? 1.0f : 0.f);
  }
  uint4 o;
  o.x = pack_bf16x2(v[0], v[1]);
  o.y = pack_bf16x2(v[2], v[3]);
  o.z = pack_bf16x2(v[4], v[5]);
  o.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(xh + (b * (T + 1) + t) * TC_XH_LD + TC_XOFF + c * 8) = o;
}

// Weight slices in the order the forward kernel consumes them.  Gate g of hidden unit 64r + 16c + jj is row
// n = 64c + 16g + jj of slice r (four 16-unit chunks of 64 gate columns each: the MMAs are issued and committed chunk by
// chunk, so the epilogue of chunk c runs under the MMAs of chunk c+1); the three sigmoid gates are pre-scaled by 0.5
// (sigmoid(z) = 0.5*tanh(z/2) + 0.5).
__device__ __forceinline__ void pack_weights_body(int bid, int I, const float* __restrict__ W, const float* __restrict__ U,
                                    const float* __restrict__ bias, __nv_bfloat16* __restrict__ Up,
                                    __nv_bfloat16* __restrict__ Wp, float* __restrict__ biasp) {
  const int H = TC_H;
  const long idx = (long)bid * blockDim.x + threadIdx.x;
  if (idx < (long)4 * H * H) {          // Up: [4][256][256]
    const int k = (int)(idx % H);
    const int n = (int)((idx / H) % TC_NSL);
    const int r = (int)(idx / ((long)H * TC_NSL));
    const int g = (n % 64) / 16, j = (n / 64) * 16 + n % 16;
    const float sc = (g == 2) ? 1.0f : 0.5f;
    Up[idx] = __float2bfloat16(sc * U[(long)k * 4 * H + g * H + r * TC_HS + j]);
  }
  if (idx < (long)4 * H * 32) {         // Wp: [4][256][32]
    const int k = (int)(idx % 32);
    const int n = (int)((idx / 32) % TC_NSL);
    const int r = (int)(idx / (32 * TC_NSL));
    const int g = (n % 64) / 16, j = (n / 64) * 16 + n % 16;
    const float sc = (g == 2) ? 1.0f : 0.5f;
    Wp[idx] = __float2bfloat16(k < I ? sc * W[(long)k * 4 * H + g * H + r * TC_HS + j] : 0.f);
  }
  if (idx < 4 * H) {                    // biasp: [4][256]
    const int n = (int)(idx % TC_NSL), r = (int)(idx / TC_NSL);
    const int g = (n % 64) / 16, j = (n / 64) * 16 + n % 16;
    biasp[idx] = ((g == 2) ? 1.0f : 0.5f) * bias[g * H + r * TC_HS + j];
  }
}

// =============================================================================================
// Persistent forward recurrence
// =============================================================================================
struct FwdParams {
  int B, T, n_iters, n_clusters, k16_x, n_tiles_cap;
  __nv_bfloat16* xh;
  __nv_bfloat16* gates;   // null: do not save
  __nv_bfloat16* cst;     // null: do not save
  const float* biasp;
  long long* trace;       // debug (LFMQ_TRACE_FWD=1): clock64 stamps of CTA 0, every third step
  unsigned int* head_progress;   // null, or per row tile (HP_CSTRIDE apart): steps whose h_t is in global memory
};

constexpr int HP_CSTRIDE = 32;   // head_progress counters one 128-byte line apart

#define FWD_TRACE(role, t, pt)                                                        \
  do {                                                                                \
    if (p.trace && blockIdx.x == 0 && (t) % 3 == 0) p.trace[((role) * 16 + (t) / 3) * 8 + (pt)] = clock64(); \
  } while (0)

constexpr int FWD_EPI_WARPS = 8;                          // 4 TMEM lane quadrants x 2 column halves
constexpr int FWD_THREADS = 32 * (2 + FWD_EPI_WARPS);     // producer + MMA + epilogue = 320
// h_t is published with one 32-byte STG per thread and chunk; one staged TMA store per CTA was slower
// (profiles/r02_time_c31_fwd_tma_publish.txt)
constexpr uint32_t SM_U = 0;                 // 4 k-blocks x [256 x 128 B]
constexpr uint32_t SM_W = 131072;            // [256 x 64 B]
constexpr uint32_t SM_H0 = 147456;           // 4 k-blocks x [128 x 128 B]
constexpr uint32_t SM_X0 = 212992;           // [128 x 64 B]
constexpr uint32_t SM_BIAS = 221184;
constexpr uint32_t SM_BARS = 222208;
constexpr uint32_t FWD_SMEM = SM_BARS + 256 + 1024;   // + alignment slack

struct FwdBars {
  uint64_t w_full, x_full, x_empty, h_full, h_written;
  uint64_t acc_full[2][4];   // [accumulator buffer][16-unit chunk]
  uint64_t acc_free;      // deferred saved-state stores have drained the staging TMEM buffer
  uint64_t tma_issued;    // producer -> epilogue: the fetch of h for the next step has been issued
  uint32_t tmem_base;
};

// SAVE: training (gates / cell states kept for BPTT).  A template parameter so that the predict kernel carries none of
// the saved-state logic.
template <bool SAVE>
__global__ void __launch_bounds__(FWD_THREADS, 1)
    lstm_fwd_tc_kernel(FwdParams p, const __grid_constant__ CUtensorMap tm_h, const __grid_constant__ CUtensorMap tm_x,
                       const __grid_constant__ CUtensorMap tm_u, const __grid_constant__ CUtensorMap tm_w) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  FwdBars* bars = reinterpret_cast<FwdBars*>(smem + SM_BARS);
  float* bias_s = reinterpret_cast<float*>(smem + SM_BIAS);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int cid = blockIdx.x / TC_NC;

  if (tid == 0) {
    mbar_init(&bars->w_full, 1);
    mbar_init(&bars->x_full, 1);
    mbar_init(&bars->x_empty, 1);
    mbar_init(&bars->h_full, 1);
    mbar_init(&bars->h_written, TC_NC);
    for (int i = 0; i < 2; ++i)
      for (int c = 0; c < 4; ++c) mbar_init(&bars->acc_full[i][c], 1);
    mbar_init(&bars->acc_free, 32 * FWD_EPI_WARPS);
    mbar_init(&bars->tma_issued, 1);
    fence_mbar_init();
  }
  if (tid < TC_NSL) bias_s[tid] = p.biasp[rank * TC_NSL + tid];
  if (warp == 1) tmem_alloc(&bars->tmem_base, 512);
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();          // peers' barriers are initialised before anyone multicasts / arrives remotely
  tcgen05_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const int T = p.T;
  // Programmatic dependent launch: everything above and the weight slice (packed two kernels ago) do not depend on the
  // preceding kernel (xh_fill_x); the 144 KB weight load overlaps its tail.
  if (!(warp == 0 && lane == 0)) pdl_sync();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(&bars->w_full, 131072 + 16384);
      for (int kb = 0; kb < 4; ++kb) tma_load_2d(smem + SM_U + kb * 32768, &tm_u, &bars->w_full, kb * 64, rank * TC_NSL);
      tma_load_2d(smem + SM_W, &tm_w, &bars->w_full, 0, rank * TC_NSL);
      pdl_sync();
      uint8_t* hbuf = smem + SM_H0;
      uint8_t* xbuf = smem + SM_X0;
      uint32_t n_hw = 0, n_xe = 0;
      for (int it = 0; it < p.n_iters; ++it) {
        const int b0 = (it * p.n_clusters + cid) * 128;
        for (int t = 0; t < T; ++t) {
          if (it > 0 || t > 0) mbar_wait(&bars->x_empty, (n_xe++) & 1);
          FWD_TRACE(0, t, 0);
          mbar_arrive_expect_tx(&bars->x_full, 8192);
          tma_load_2d(xbuf, &tm_x, &bars->x_full, t * TC_XH_LD + TC_XOFF, b0);
          if (t >= 1) {
            mbar_wait_cluster(&bars->h_written, (n_hw++) & 1);   // all 4 slices of h_{t-1} are in global memory
            FWD_TRACE(0, t, 1);
            fence_proxy_async_global();
            mbar_arrive_expect_tx(&bars->h_full, 65536);
            for (int kb = 0; kb < 4; ++kb)
              tma_load_2d_mcast(hbuf + kb * 16384 + rank * 4096, &tm_h, &bars->h_full, t * TC_XH_LD + kb * 64,
                                b0 + 32 * (int)rank, 0xF);
            FWD_TRACE(0, t, 2);
            if (SAVE) mbar_arrive(&bars->tma_issued);
            // h_{t-1} of all 4 CTAs is in global memory (acquired above): count it for the paced head.  A gpu-scope
            // release, cumulative over the cluster barrier, from the one thread with a step of slack after it
            if (p.head_progress && rank == 0)
              red_release_gpu_add(p.head_progress + (it * p.n_clusters + cid) * HP_CSTRIDE, 1u);
          }
        }
        mbar_wait_cluster(&bars->h_written, (n_hw++) & 1);       // phase of step T-1 (keeps parities aligned)
        if (p.head_progress && rank == 0)
          red_release_gpu_add(p.head_progress + (it * p.n_clusters + cid) * HP_CSTRIDE, 1u);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, 64, false, false);      // one 16-unit chunk = 64 gate columns
      mbar_wait(&bars->w_full, 0);
      uint32_t n_xf = 0, n_hf = 0;
      for (int it = 0; it < p.n_iters; ++it) {
        for (int t = 0; t < T; ++t) {
          const uint32_t g = (uint32_t)(it * T + t);
          const uint32_t acc = tmem + (g & 1) * 256;
          mbar_wait(&bars->x_full, (n_xf++) & 1);
          // training: acc[g&1] doubled as the staging buffer of step g-1's saved gates / cell states
          if (SAVE && g > 0) mbar_wait(&bars->acc_free, (g - 1) & 1);
          FWD_TRACE(1, t, 0);
          tcgen05_fence_after();
          // x part of all four chunks first (it does not wait for h), then the h part chunk by chunk, each chunk
          // committed on its own barrier: the epilogue of chunk c overlaps the MMAs of chunks c+1..
          for (int c = 0; c < 4; ++c)
            for (int k16 = 0; k16 < p.k16_x; ++k16) {
              const uint64_t da = make_smem_desc(smem_u32(smem + SM_X0) + k16 * 32, 0, 512, LAYOUT_SW64);
              const uint64_t db = make_smem_desc(smem_u32(smem + SM_W + c * 4096) + k16 * 32, 0, 512, LAYOUT_SW64);
              umma_f16(acc + c * 64, da, db, idesc, k16 > 0);
            }
          umma_commit(&bars->x_empty);
          if (t == 0) {
            for (int c = 0; c < 4; ++c) umma_commit(&bars->acc_full[g & 1][c]);
          } else {
            mbar_wait(&bars->h_full, (n_hf++) & 1);
            FWD_TRACE(1, t, 1);
            tcgen05_fence_after();
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
              for (int kb = 0; kb < 4; ++kb)
#pragma unroll
                for (int k16 = 0; k16 < 4; ++k16) {
                  const uint64_t da = make_smem_desc(smem_u32(smem + SM_H0 + kb * 16384) + k16 * 32, 0, 1024, LAYOUT_SW128);
                  const uint64_t db = make_smem_desc(smem_u32(smem + SM_U + kb * 32768 + c * 8192) + k16 * 32, 0, 1024,
                                                     LAYOUT_SW128);
                  umma_f16(acc + c * 64, da, db, idesc, 1);
                }
              umma_commit(&bars->acc_full[g & 1][c]);
            }
            FWD_TRACE(1, t, 2);
          }
        }
      }
    }
  } else {
    // ===================== epilogue: gates, cell update, h exchange =====================
    const int half = (warp - 2) / 4;        // this warp takes the 16-unit chunks half and half + 2 of the CTA's 64 units
    const int q = warp & 3;                 // TMEM lane quadrant this warp may touch
    const int m = q * 32 + lane;            // row of the 128-row tile
    const bool leader = (warp == 2) && lane == 0;
    uint32_t n_ti = 0;                      // phases of tma_issued consumed (one per step that has a successor)
    float cstate[32];
    for (int it = 0; it < p.n_iters; ++it) {
      const int tile_c = it * p.n_clusters + cid;
      const long b = (long)tile_c * 128 + m;
      const bool valid = b < p.B;
#pragma unroll
      for (int j = 0; j < 32; ++j) cstate[j] = 0.f;
      for (int t = 0; t < T; ++t) {
        const uint32_t g = (uint32_t)(it * T + t);
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const uint32_t taddr_other = tmem + lane_addr + ((g + 1) & 1) * 256 + half * 80;
        // saved state, SoA at 32-byte granularity: [(t, tile, 32-unit block fr, quadrant)][piece = gate*2 + h16][lane],
        // unit = 32 fr + 16 h16 + e.  Chunk c = half + 2 jb of this CTA is fr = 2 rank + jb, h16 = half.
        const long wblk0 = (((long)t * p.n_tiles_cap + tile_c) * 8 + 2 * (int)rank) * 4 + q;      // jb = 0; jb = 1: + 4
        __nv_bfloat16* grow = SAVE ? p.gates + (wblk0 * 8 * 32 + lane) * 16 + half * 512 : nullptr;   // + gate*1024 (+ jb*4*8*512)
        __nv_bfloat16* crow = SAVE ? p.cst + (wblk0 * 2 * 32 + lane) * 16 + half * 512 : nullptr;     // (+ jb*4*2*512)
#pragma unroll
        for (int jb = 0; jb < 2; ++jb) {
          const int c = half + 2 * jb;            // 16-unit chunk of this CTA's 64 hidden units
          mbar_wait(&bars->acc_full[g & 1][c], (g >> 1) & 1);
          if (leader && jb == 0) FWD_TRACE(2, t, 0);
          tcgen05_fence_after();
          const uint32_t taddr = tmem + lane_addr + (g & 1) * 256 + c * 64;
          __nv_bfloat16* hrow = p.xh + (b * (T + 1) + (t + 1)) * TC_XH_LD + rank * TC_HS + c * 16;
          uint32_t vi[16], vf[16], vg[16], vo[16];
          tmem_ld_32x32b_x16(taddr + 0, vi);
          tmem_ld_32x32b_x16(taddr + 16, vf);
          tmem_ld_32x32b_x16(taddr + 32, vg);
          tmem_ld_32x32b_x16(taddr + 48, vo);
          tmem_ld_wait();
          uint32_t ph[8], pi[8], pf[8], pg[8], po[8];
          float cn[16];
          const float* bs = bias_s + c * 64;
#pragma unroll
          for (int jj = 0; jj < 16; jj += 2) {
            float hv[2], iv[2], fv[2], gv[2], ov[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int j = jb * 16 + jj + u;
              const float gi = fmaf(0.5f, tanh_approx(__uint_as_float(vi[jj + u]) + bs[jj + u]), 0.5f);
              const float gf = fmaf(0.5f, tanh_approx(__uint_as_float(vf[jj + u]) + bs[16 + jj + u]), 0.5f);
              const float gg = tanh_approx(__uint_as_float(vg[jj + u]) + bs[32 + jj + u]);
              const float go = fmaf(0.5f, tanh_approx(__uint_as_float(vo[jj + u]) + bs[48 + jj + u]), 0.5f);
              const float cc = fmaf(gf, cstate[j], gi * gg);
              cstate[j] = cc;
              cn[jj + u] = cc;
              hv[u] = go * tanh_approx(cc);
              iv[u] = gi; fv[u] = gf; gv[u] = gg; ov[u] = go;
            }
            ph[jj / 2] = pack_bf16x2(hv[0], hv[1]);
            pi[jj / 2] = pack_bf16x2(iv[0], iv[1]);
            pf[jj / 2] = pack_bf16x2(fv[0], fv[1]);
            pg[jj / 2] = pack_bf16x2(gv[0], gv[1]);
            po[jj / 2] = pack_bf16x2(ov[0], ov[1]);
          }
          if (valid) st_global_v8(hrow, ph);   // one full 32-byte sector per store (STG.256)
          if (SAVE) {
            // Saved gates / cell states are not needed by the h exchange: park them in the idle accumulator
            // buffer (TMEM) and write them to HBM after the publish, off the per-step critical path.
            const uint32_t tst = taddr_other + jb * 40;
            uint32_t cu[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) cu[e] = pack_bf16x2(cn[2 * e], cn[2 * e + 1]);
            tmem_st_32x32b_x8(tst, pi);
            tmem_st_32x32b_x8(tst + 8, pf);
            tmem_st_32x32b_x8(tst + 16, pg);
            tmem_st_32x32b_x8(tst + 24, po);
            tmem_st_32x32b_x8(tst + 32, cu);
          }
        }
        if (SAVE) tmem_st_wait();
        tcgen05_fence_before();
        if (leader) FWD_TRACE(2, t, 1);
        // Publish this CTA's h slice: CTA-level barrier over the 256 epilogue threads, then 4 lanes of the leader
        // warp arrive (release.cluster, cumulative over the barrier) on the 4 CTAs' h_written barriers in parallel.
        // Readers acquire at cluster scope and cross into the async proxy before their TMA loads.
        named_bar_sync(1, 32 * FWD_EPI_WARPS);
        if (leader) FWD_TRACE(2, t, 4);
        if (warp == 2 && lane < TC_NC)
          mbar_arrive_cluster(mapa_u32(smem_u32(&bars->h_written), (uint32_t)lane));
        if (SAVE) {
          // Saved state of this step, parked in the idle accumulator buffer.  All CTAs reach this point together, so
          // writing the whole 80 KB per CTA at once is a ~3 K-cycle burst at full HBM write bandwidth: it outlasts the
          // publish, and the producer's proxy fence + TMA issue for the next step then queue behind it (clock64 trace:
          // 1.5 K cycles instead of 0.3 K without saved state).  So: first half now (over before the producer needs to
          // fence), second half out of TMEM into registers -- the MMA may have the staging buffer back -- and to global
          // only once the producer has issued the next step's h fetch.
          tcgen05_fence_after();
          uint32_t sg[32], sc[8];
          tmem_ld_32x32b_x32(taddr_other, sg);
          tmem_ld_32x32b_x8(taddr_other + 32, sc);
          tmem_ld_wait();
          if (valid) {      // chunk jb = 0 (32-unit block fr = 2 rank)
            st_global_v8(grow + 0 * 1024, sg);
            st_global_v8(grow + 1 * 1024, sg + 8);
            st_global_v8(grow + 2 * 1024, sg + 16);
            st_global_v8(grow + 3 * 1024, sg + 24);
            st_global_v8(crow, sc);
          }
          tmem_ld_32x32b_x32(taddr_other + 40, sg);
          tmem_ld_32x32b_x8(taddr_other + 40 + 32, sc);
          tmem_ld_wait();
          tcgen05_fence_before();
          mbar_arrive(&bars->acc_free);
          if (t < T - 1) mbar_wait(&bars->tma_issued, (n_ti++) & 1);
          if (valid) {      // chunk jb = 1 (32-unit block fr = 2 rank + 1: 4 quadrant blocks further)
            __nv_bfloat16* grow1 = grow + 4L * 8 * 512;
            st_global_v8(grow1 + 0 * 1024, sg);
            st_global_v8(grow1 + 1 * 1024, sg + 8);
            st_global_v8(grow1 + 2 * 1024, sg + 16);
            st_global_v8(grow1 + 3 * 1024, sg + 24);
            st_global_v8(crow + 4L * 2 * 512, sc);
          }
        }
        if (leader) FWD_TRACE(2, t, 5);
      }
    }
  }
  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();          // nobody leaves while peers may still multicast into / arrive on this CTA
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// =============================================================================================
// Fused head: BN(inference affine) -> Dropout -> Dense -> weighted-MSE loss -> (training) all head gradients
// and dLoss/dh.  One warp per [b,t] row, H = 256 (8 hidden units per lane), n_outputs <= 16.
// (models/point_estimate/rnn_point_estimate.py:88-89,105; model_utils/losses.py:55-135; SURVEY App. A.2-A.4)
// =============================================================================================
struct HeadParams {
  int B, T, O, target_idx, train;
  const __nv_bfloat16* xh;
  const float *gamma, *beta, *mean, *var;
  float eps;
  const float *Wo, *bo;
  const float* y;
  const float* denom;
  float p1, p2;
  int use_dropout;
  DropoutKey key;
  int64_t row0;
  float* preds;
  __nv_bfloat16* dhout;
  float* dpred;         // [B*T][16] dLoss/dpred (training), consumed by head_wgrad_kernel
  float* partial;       // [gridDim.x][HEAD_PART]
  long long* trace;     // debug (LFMQ_TRACE_HEAD=1): clock64 stamps of CTA 0, first 8 tiles
};

#define HEAD_TRACE(role, n, pt)                                                                       \
  do {                                                                                                \
    if (p.trace && blockIdx.x == 0 && (n) < 8) p.trace[((role) * 8 + (n)) * 8 + (pt)] = clock64();    \
  } while (0)

constexpr int HEAD_PART = 2 * TC_H + TC_OPAD + 16;   // dgamma | dbeta | dbo | s0 s1 s2 (per CTA of the fused pass)
constexpr int HEAD_THREADS = 256;
constexpr int HWG_PART = TC_H * TC_OPAD;              // dWo partial per CTA of the weight-gradient pass
constexpr int HWG_ROWS = 32;                          // rows staged per tile

// Thread-per-row head over TMA-staged tiles: a CTA takes 128 windows of one time step (the 128 x 256 bf16 h tile
// arrives as four SWIZZLE_128B boxes), every thread owns one row: y = Dropout(BN(h)) on the fly, pred = y*Wo + bo
// with Wo broadcast from shared memory (no cross-lane traffic), loss terms, dLoss/dpred, dy = dpred*Wo^T, dLoss/dh
// written in the backward kernel's SoA layout; dgamma/dbeta need a cross-row sum per column, done with a 31-shuffle
// reduce-scatter per group of 32 columns.
constexpr int HROWS_SMEM = 65536 + 1024 + 256;

template <bool TRAIN>
__global__ void __launch_bounds__(128, 2) head_rows_kernel(HeadParams p, const __grid_constant__ CUtensorMap tm_h,
                                                          int n_btiles, int n_tiles_cap) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar = reinterpret_cast<uint64_t*>(tile + 65536);
  __shared__ __align__(16) float Wo_s[TC_H * TC_OPAD];
  __shared__ __align__(16) float bn_s[4][TC_H];      // gamma*inv | beta - gamma*mean*inv | mean | inv
  __shared__ float red_s[HEAD_PART];
  const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
  for (int j = tid; j < TC_H; j += 128) {
    const float iv = 1.0f / sqrtf(p.var[j] + p.eps);
    bn_s[0][j] = p.gamma[j] * iv;
    bn_s[1][j] = p.beta[j] - p.gamma[j] * p.mean[j] * iv;
    bn_s[2][j] = p.mean[j];
    bn_s[3][j] = iv;
  }
  for (int i = tid; i < TC_H * TC_OPAD; i += 128) {
    const int j = i / TC_OPAD, k = i % TC_OPAD;
    Wo_s[i] = (k < p.O) ? p.Wo[j * p.O + k] : 0.f;
  }
  for (int i = tid; i < HEAD_PART; i += 128) red_s[i] = 0.f;
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
  float accbo[TC_OPAD];
#pragma unroll
  for (int k = 0; k < TC_OPAD; ++k) accbo[k] = 0.f;
  const int sw = tid & 7;
  const int nq = TC_H / 4;
  uint32_t phase = 0;
  const int n_tiles = p.T * n_btiles;
  for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
    const int t = ti / n_btiles, bt = ti % n_btiles;
    const long b = (long)bt * 128 + tid;
    const bool valid = b < p.B;
    if (tid == 0) {
      mbar_arrive_expect_tx(bar, 65536);
      for (int kb = 0; kb < 4; ++kb)
        tma_load_2d(tile + kb * 16384, &tm_h, bar, (t + 1) * TC_XH_LD + kb * 64, bt * 128);
    }
    const long r = b * p.T + t;
    float yt[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) yt[k] = 0.f;
    if (p.y && valid) {
      for (int k = 0; k < p.O; ++k) yt[k] = p.y[r * p.O + k];
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    const uint8_t* hrow = tile + tid * 128;
    float pr[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) pr[k] = (k < p.O) ? p.bo[k] : 0.f;
#pragma unroll 4
    for (int c = 0; c < 32; ++c) {
      const uint4 raw = *reinterpret_cast<const uint4*>(hrow + (c >> 3) * 16384 + (((c & 7) ^ sw) << 4));
      const uint32_t hw[4] = {raw.x, raw.y, raw.z, raw.w};
      float dm[8];
      if (p.use_dropout) {
        const uint64_t qbase = ((uint64_t)(p.row0 + b) * p.T + t) * nq + c * 2;
        dropout_quad(p.key, qbase, dm);
        dropout_quad(p.key, qbase + 1, dm + 4);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) dm[e] = 1.f;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int j = c * 8 + e;
        const float hv = (e & 1) ? bf16_hi(hw[e >> 1]) : bf16_lo(hw[e >> 1]);
        const float yv = fmaf(bn_s[0][j], hv, bn_s[1][j]) * dm[e];
        const float4* w4 = reinterpret_cast<const float4*>(Wo_s + j * TC_OPAD);
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
    if (p.preds && valid) {
      for (int k = 0; k < p.O; ++k) p.preds[r * p.O + k] = pr[k];
    }
    if (p.y) {
      bool any = false;
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) any |= (yt[k] != 0.0f);          // losses.py:72
      const float mk = (any && valid) ? 1.f : 0.f;
      const bool last = (t == p.T - 1);
      float dp[TC_OPAD];
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) {
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
        if (valid) {
#pragma unroll
          for (int k4 = 0; k4 < TC_OPAD; k4 += 4)
            *reinterpret_cast<float4*>(p.dpred + r * TC_OPAD + k4) = make_float4(dp[k4], dp[k4 + 1], dp[k4 + 2], dp[k4 + 3]);
        }
        // dLoss/dh in the backward kernel's layout: [t][tile][rank r'][warp][chunk][lane][16]
        __nv_bfloat16* dh_base = p.dhout + ((((long)t * n_tiles_cap + bt) * 4) * 4 + wq) * 4 * 32 * 16 + lane * 16;
#pragma unroll 1
        for (int grp = 0; grp < 8; ++grp) {          // 32 columns per group
          float dd[32], gd[32];
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            const int c = grp * 4 + cc;
            const uint4 raw = *reinterpret_cast<const uint4*>(hrow + (c >> 3) * 16384 + (((c & 7) ^ sw) << 4));
            const uint32_t hw[4] = {raw.x, raw.y, raw.z, raw.w};
            float dm[8];
            if (p.use_dropout) {
              const uint64_t qbase = ((uint64_t)(p.row0 + b) * p.T + t) * nq + c * 2;
              dropout_quad(p.key, qbase, dm);
              dropout_quad(p.key, qbase + 1, dm + 4);
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) dm[e] = 1.f;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int j = c * 8 + e;
              const float hv = (e & 1) ? bf16_hi(hw[e >> 1]) : bf16_lo(hw[e >> 1]);
              const float4* w4 = reinterpret_cast<const float4*>(Wo_s + j * TC_OPAD);
              float sacc = 0.f;
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const float4 w = w4[kk];
                sacc = fmaf(dp[4 * kk + 0], w.x, sacc);
                sacc = fmaf(dp[4 * kk + 1], w.y, sacc);
                sacc = fmaf(dp[4 * kk + 2], w.z, sacc);
                sacc = fmaf(dp[4 * kk + 3], w.w, sacc);
              }
              const float d_ = sacc * dm[e];                       // through Dropout
              dd[cc * 8 + e] = d_;
              gd[cc * 8 + e] = d_ * (hv - bn_s[2][j]) * bn_s[3][j];
            }
          }
          // dLoss/dh = dd * gamma * inv -> two 16-unit chunks of this group
          if (valid) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t pk[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int jj = hh * 16 + 2 * e;
                pk[e] = pack_bf16x2(dd[jj] * bn_s[0][grp * 32 + jj], dd[jj + 1] * bn_s[0][grp * 32 + jj + 1]);
              }
              const int c16 = grp * 2 + hh;                         // 16-unit chunk 0..15: rank r' = c16/4, chunk c16%4
              st_global_v8(dh_base + ((long)(c16 >> 2) * 4 * 4 + (c16 & 3)) * 32 * 16, pk);
            }
          }
          // column sums over the warp's 32 rows: reduce-scatter butterfly, lane l ends with column perm(l)
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const bool up = (lane & off) != 0;
              const float sd = up ? dd[i] : dd[i + off];
              const float kd = up ? dd[i + off] : dd[i];
              dd[i] = kd + __shfl_xor_sync(0xffffffffu, sd, off);
              const float sg = up ? gd[i] : gd[i + off];
              const float kg = up ? gd[i + off] : gd[i];
              gd[i] = kg + __shfl_xor_sync(0xffffffffu, sg, off);
            }
          }
          // lane's column within the group: bit b of lane selects +2^b  (lane bit4 -> +16 ... bit0 -> +1)
          atomicAdd(&red_s[TC_H + grp * 32 + lane], dd[0]);
          atomicAdd(&red_s[grp * 32 + lane], gd[0]);
        }
      }
    }
    __syncthreads();        // everyone is done with the tile before it is overwritten
  }
  if (p.y) {
    // block-level sums of the loss terms and dbo
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) accbo[k] = warp_sum(accbo[k]);
    if (lane == 0) {
      atomicAdd(&red_s[2 * TC_H + TC_OPAD + 0], s0);
      atomicAdd(&red_s[2 * TC_H + TC_OPAD + 1], s1);
      atomicAdd(&red_s[2 * TC_H + TC_OPAD + 2], s2);
      if (TRAIN)
        for (int k = 0; k < TC_OPAD; ++k) atomicAdd(&red_s[2 * TC_H + k], accbo[k]);
    }
    __syncthreads();
    for (int i = tid; i < HEAD_PART; i += 128) p.partial[(long)i * gridDim.x + blockIdx.x] = red_s[i];
  }
}

// Tensor-core head (dropout off): with y = a*h + b (BN inference affine) the Dense layer folds to
//   pred = h * (diag(a) Wo) + (bo + b Wo)
// a tcgen05 MMA on the TMA-staged h tile (K-major SW128, exactly the layout the recurrence uses): 16 x (M128 N16 K16).
// Threads own one row each for the loss terms and dpred, staged as a 128 x 32 bf16 tile (SW64).  Training: that tile
// feeds h^T dpred (MN-major MMAs, accumulated in TMEM across tiles -> dWo, dgamma) and goes to HBM by TMA store for the
// backward recurrence, which forms dLoss/dh = dpred (Wo a)^T on its own tensor cores; colsum(dpred) -> dbo, dbeta.
struct HeadTcWeights {
  const __nv_bfloat16* WoTp;   // [16][256]  a_j * Wo[j][n]
  const float* bop;            // [16]       bo + sum_j b_j Wo[j][k]
};

__device__ __forceinline__ void pack_head_body(int bid, int O, const float* __restrict__ Wo, const float* __restrict__ bo,
                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                 const float* __restrict__ mean, const float* __restrict__ var, float eps,
                                 __nv_bfloat16* __restrict__ WoTp, __nv_bfloat16* __restrict__ WoSp,
                                 float* __restrict__ bop) {
  const int idx = bid * blockDim.x + threadIdx.x;
  if (idx < TC_OPAD * TC_H) {
    const int n = idx / TC_H, j = idx % TC_H;
    const float a = gamma[j] / sqrtf(var[j] + eps);
    WoTp[idx] = __float2bfloat16(n < O ? a * Wo[j * O + n] : 0.f);
  }
  if (idx < TC_H * 32) {
    const int j = idx / 32, k = idx % 32;
    WoSp[idx] = __float2bfloat16(k < O ? Wo[j * O + k] * gamma[j] / sqrtf(var[j] + eps) : 0.f);
  }
  // folded bias: block k (< 16) reduces over its 256 threads = 256 hidden units
  if (bid < TC_OPAD) {
    __shared__ float red[8];
    const int k = bid, j = threadIdx.x;
    float v = 0.f;
    if (k < O) {
      const float iv = 1.0f / sqrtf(var[j] + eps);
      v = (beta[j] - gamma[j] * mean[j] * iv) * Wo[j * O + k];
    }
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = (k < O) ? bo[k] : 0.f;
      for (int w = 0; w < 8; ++w) t += red[w];
      bop[k] = t;
    }
  }
}

// Ubk[r][n][k'] = U[n][g*H + 64r + 16jb + jj], k' = 64jb + 16g + jj   (K-slices of U for the backward recurrence)
__device__ __forceinline__ void pack_ubk_body(int bid, const float* __restrict__ U, __nv_bfloat16* __restrict__ Ubk) {
  const long idx = (long)bid * blockDim.x + threadIdx.x;
  if (idx >= (long)4 * TC_H * TC_H) return;
  const int kp = (int)(idx % 256);
  const int n = (int)((idx / 256) % TC_H);
  const int r = (int)(idx / (256 * TC_H));
  const int jb = kp / 64, g = (kp % 64) / 16, jj = kp % 16;
  Ubk[idx] = __float2bfloat16(U[(long)n * 4 * TC_H + g * TC_H + 64 * r + 16 * jb + jj]);
}

// All weight repacking of one optimizer step in ONE launch: block ranges [0,nb_w) forward slices, [nb_w,nb_w+nb_h)
// head, the rest the backward K-slices (nb_u = 0 on a forward-only handle).
struct PackArgs {
  int I, O, nb_w, nb_h, nb_u;
  float eps;
  const float *W, *U, *bias, *Wo, *bo, *gamma, *beta, *mean, *var;
  __nv_bfloat16 *Up, *Wp, *Ubk, *WoTp, *WoSp;
  float *biasp, *bop;
};

__global__ void __launch_bounds__(256) pack_all_kernel(PackArgs a) {
  pdl_sync();
  const int bid = blockIdx.x;
  if (bid < a.nb_w) {
    pack_weights_body(bid, a.I, a.W, a.U, a.bias, a.Up, a.Wp, a.biasp);
  } else if (bid < a.nb_w + a.nb_h) {
    pack_head_body(bid - a.nb_w, a.O, a.Wo, a.bo, a.gamma, a.beta, a.mean, a.var, a.eps, a.WoTp, a.WoSp, a.bop);
  } else {
    pack_ubk_body(bid - a.nb_w - a.nb_h, a.U, a.Ubk);
  }
}

constexpr uint32_t HT_TILE = 0;            // 4 k-blocks x [128 x 128 B]
constexpr uint32_t HT_WOT = 65536;         // 4 k-blocks x [16 x 128 B]
// (73728 .. 90111: unused since dLoss/dh moved to the backward kernel; kept so the tile offsets stay 1024-aligned)
constexpr uint32_t HT_DP = 90112;          // [128 x 64 B]
constexpr uint32_t HT_BARS = 98304;
constexpr int HT_SMEM = HT_BARS + 128 + 1024;
constexpr int HT_THREADS = 160;            // warp 0: TMA + MMA issue, warps 1-4: one row per thread

struct HtBars {
  uint64_t wt_full, tile_full, pred_full, dp_full, dp_free, tile_free, w_done;
  uint32_t tmem_base;
};

template <bool TRAIN>
__global__ void __launch_bounds__(HT_THREADS, 2)
    head_tc_kernel(HeadParams p, HeadTcWeights w, const __grid_constant__ CUtensorMap tm_h,
                   const __grid_constant__ CUtensorMap tm_wot, const __grid_constant__ CUtensorMap tm_dpb, int n_btiles, int n_tiles_cap,
                   float* __restrict__ wpartial) {
  pdl_sync();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  HtBars* bars = reinterpret_cast<HtBars*>(smem + HT_BARS);
  __shared__ __align__(16) float bn_s[3][TC_H];      // gamma*inv | mean | inv
  __shared__ float red_s[HEAD_PART];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int j = tid; j < TC_H; j += HT_THREADS) {
    const float iv = 1.0f / sqrtf(p.var[j] + p.eps);
    bn_s[0][j] = p.gamma[j] * iv;
    bn_s[1][j] = p.mean[j];
    bn_s[2][j] = iv;
  }
  for (int i = tid; i < HEAD_PART; i += HT_THREADS) red_s[i] = 0.f;
  // zero the dpred staging tile once (padding columns stay zero)
  for (int i = tid; i < 128 * 64 / 16; i += HT_THREADS) reinterpret_cast<uint4*>(smem + HT_DP)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    mbar_init(&bars->wt_full, 1);
    mbar_init(&bars->tile_full, 1);
    mbar_init(&bars->pred_full, 1);
    mbar_init(&bars->dp_full, 128);
    mbar_init(&bars->dp_free, 1);
    mbar_init(&bars->tile_free, 128);
    mbar_init(&bars->w_done, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&bars->tmem_base, 256);
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const uint32_t acc_p = tmem;             // 16 columns
  const uint32_t acc_w = tmem + 160;       // 2 x 16 columns: sum over this CTA's tiles of h^T dpred (rows = hidden unit)
  const int n_tiles = p.T * n_btiles;

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(&bars->wt_full, 8192);
      for (int kb = 0; kb < 4; ++kb) tma_load_2d(smem + HT_WOT + kb * 2048, &tm_wot, &bars->wt_full, kb * 64, 0);
      mbar_wait(&bars->wt_full, 0);
      const uint32_t idesc_p = make_idesc_bf16(128, 16, false, false);
      uint32_t n = 0;
      for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++n) {
        const int t = ti / n_btiles, bt = ti % n_btiles;
        if (n > 0) mbar_wait(TRAIN ? &bars->dp_free : &bars->tile_free, (n - 1) & 1);
        HEAD_TRACE(0, n, 0);
        mbar_arrive_expect_tx(&bars->tile_full, 65536);
        for (int kb = 0; kb < 4; ++kb)
          tma_load_2d(smem + HT_TILE + kb * 16384, &tm_h, &bars->tile_full, (t + 1) * TC_XH_LD + kb * 64, bt * 128);
        mbar_wait(&bars->tile_full, n & 1);
        HEAD_TRACE(0, n, 1);
        tcgen05_fence_after();
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
          for (int k16 = 0; k16 < 4; ++k16) {
            const uint64_t da = make_smem_desc(smem_u32(smem + HT_TILE + kb * 16384) + k16 * 32, 0, 1024, LAYOUT_SW128);
            const uint64_t db = make_smem_desc(smem_u32(smem + HT_WOT + kb * 2048) + k16 * 32, 0, 1024, LAYOUT_SW128);
            umma_f16(acc_p, da, db, idesc_p, (kb | k16) != 0);
          }
        umma_commit(&bars->pred_full);
        if (TRAIN) {
          mbar_wait(&bars->dp_full, n & 1);
          HEAD_TRACE(0, n, 2);
          tcgen05_fence_after();
          // the staged dLoss/dpred tile also goes to HBM as it is (128 x 64 B, SW64): the backward recurrence adds
          // dpred (Wo gamma inv)^T for its own hidden units on its tensor cores
          tma_store_2d(&tm_dpb, smem + HT_DP, 0, (t * n_tiles_cap + bt) * 128);
          bulk_commit_group();
          // dWo' += h^T dpred: A = the h tile read MN-major (hidden unit = M), B = the dpred tile read MN-major,
          // K = the 128 rows.
          {
            const uint32_t idesc_w = make_idesc_bf16(128, 16, true, true);
#pragma unroll
            for (int mb = 0; mb < 2; ++mb)
#pragma unroll
              for (int k16 = 0; k16 < 8; ++k16) {
                const uint64_t wa = make_smem_desc(smem_u32(smem + HT_TILE + 2 * mb * 16384) + k16 * 2048, 16384, 1024,
                                                   LAYOUT_SW128);
                const uint64_t wb = make_smem_desc(smem_u32(smem + HT_DP) + k16 * 1024, 0, 512, LAYOUT_SW64);
                umma_f16(acc_w + mb * 16, wa, wb, idesc_w, (n > 0 || k16 > 0) ? 1u : 0u);
              }
          }
          bulk_wait_group_read0();          // the store has read the dpred tile
          umma_commit(&bars->dp_free);      // ... and the h^T dpred MMAs are done with it and with the h tile
          HEAD_TRACE(0, n, 3);
        }
      }
      if (TRAIN) {
        umma_commit(&bars->w_done);
        bulk_wait_group0();
      }
    }
  } else {
    const int m = tid - 32;                 // row of the tile
    const int wq = warp & 3;                // TMEM lane quadrant of this warp
    const int mrow = wq * 32 + lane;        // row this thread can reach in TMEM == row it owns
    (void)m;
    const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
    float c_all = 0.f, c_last = 0.f, c_tar = 0.f;
    if (TRAIN) {
      const float Bg = p.denom[0], Mg = p.denom[1];
      c_all = (1.f - p.p1) * (1.f - p.p2) / ((float)p.O * Mg);
      c_last = (1.f - p.p1) * p.p2 / (Bg * (float)p.O);
      c_tar = p.p1 / Bg;
    }
    float bop[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) bop[k] = w.bop[k];
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    float accbo[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) accbo[k] = 0.f;
    uint32_t n = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++n) {
      const int t = ti / n_btiles, bt = ti % n_btiles;
      const long b = (long)bt * 128 + mrow;
      const bool valid = b < p.B;
      const long r = b * p.T + t;
      float yt[TC_OPAD];
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) yt[k] = 0.f;
      if (p.y && valid) {
#pragma unroll
        for (int k = 0; k < TC_OPAD; ++k)
          if (k < p.O) yt[k] = p.y[r * p.O + k];
      }
      mbar_wait(&bars->pred_full, n & 1);
      if (tid == 32) HEAD_TRACE(1, n, 0);
      tcgen05_fence_after();
      uint32_t pv[16];
      tmem_ld_32x32b_x16(acc_p + lane_addr, pv);
      tmem_ld_wait();
      float pr[TC_OPAD];
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) pr[k] = __uint_as_float(pv[k]) + bop[k];
      if (p.preds && valid) {
#pragma unroll
        for (int k = 0; k < TC_OPAD; ++k)
          if (k < p.O) p.preds[r * p.O + k] = pr[k];
      }
      if (p.y) {
        bool any = false;
#pragma unroll
        for (int k = 0; k < TC_OPAD; ++k) any |= (yt[k] != 0.0f);          // losses.py:72
        const float mk = (any && valid) ? 1.f : 0.f;
        const bool last = (t == p.T - 1);
        float dp[TC_OPAD];
#pragma unroll
        for (int k = 0; k < TC_OPAD; ++k) {
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
          if (valid && p.dpred) {        // fp32 copy: only the dropout path's SIMT weight-gradient kernel reads it
#pragma unroll
            for (int k4 = 0; k4 < TC_OPAD; k4 += 4)
              *reinterpret_cast<float4*>(p.dpred + r * TC_OPAD + k4) = make_float4(dp[k4], dp[k4 + 1], dp[k4 + 2], dp[k4 + 3]);
          }
          // dpred row -> A operand tile [128 x 64 B], SWIZZLE_64B: chunk c of row m at m*64 + ((c ^ ((m>>1)&3)) << 4)
          if (n > 0) mbar_wait(&bars->dp_free, (n - 1) & 1);     // MMAs and the TMA store are done with the previous tile
          uint8_t* drow = smem + HT_DP + mrow * 64;
          const int s64 = (mrow >> 1) & 3;
          *reinterpret_cast<uint4*>(drow + ((0 ^ s64) << 4)) =
              make_uint4(pack_bf16x2(dp[0], dp[1]), pack_bf16x2(dp[2], dp[3]), pack_bf16x2(dp[4], dp[5]), pack_bf16x2(dp[6], dp[7]));
          *reinterpret_cast<uint4*>(drow + ((1 ^ s64) << 4)) =
              make_uint4(pack_bf16x2(dp[8], dp[9]), pack_bf16x2(dp[10], dp[11]), pack_bf16x2(dp[12], dp[13]), pack_bf16x2(dp[14], dp[15]));
          fence_proxy_async_smem();
          mbar_arrive(&bars->dp_full);
          if (tid == 32) HEAD_TRACE(1, n, 1);
          // nothing else per tile: dLoss/dh is formed by the backward recurrence from the dpred tile (lstm_bwd_tc_kernel
          // <FUSED>), dgamma / dbeta by head_fold_kernel from h^T dpred and colsum(dpred)
        }
      }
      tcgen05_fence_before();
      if (!TRAIN) mbar_arrive(&bars->tile_free);
    }
    if (p.y) {
      s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) accbo[k] = warp_sum(accbo[k]);
      if (lane == 0) {
        atomicAdd(&red_s[2 * TC_H + TC_OPAD + 0], s0);
        atomicAdd(&red_s[2 * TC_H + TC_OPAD + 1], s1);
        atomicAdd(&red_s[2 * TC_H + TC_OPAD + 2], s2);
        if (TRAIN)
          for (int k = 0; k < TC_OPAD; ++k) atomicAdd(&red_s[2 * TC_H + k], accbo[k]);
      }
    }
    if (TRAIN) {
      // this CTA's h^T dpred: TMEM lane = hidden unit (mod 128), 16 columns per 128-unit block
      float* wp = wpartial + (long)blockIdx.x * HWG_PART;
      if (n > 0) {
        mbar_wait(&bars->w_done, 0);
        tcgen05_fence_after();
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(acc_w + lane_addr + mb * 16, v);
          tmem_ld_wait();
          float* o = wp + (mb * 128 + mrow) * TC_OPAD;
#pragma unroll
          for (int k4 = 0; k4 < 16; k4 += 4)
            *reinterpret_cast<float4*>(o + k4) = make_float4(__uint_as_float(v[k4]), __uint_as_float(v[k4 + 1]),
                                                             __uint_as_float(v[k4 + 2]), __uint_as_float(v[k4 + 3]));
        }
      } else {
        for (int mb = 0; mb < 2; ++mb)
          for (int k = 0; k < TC_OPAD; ++k) wp[(mb * 128 + mrow) * TC_OPAD + k] = 0.f;
      }
    }
  }
  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (p.y)
    for (int i = tid; i < HEAD_PART; i += HT_THREADS) p.partial[(long)i * gridDim.x + blockIdx.x] = red_s[i];
  if (warp == 0) tmem_dealloc(tmem, 256);
}

// dWo[j][k] = sum_r y[r][j] * dpred[r][k] with y = Dropout(BN(h)) recomputed from h: CTA tiles of 32 rows staged in
// shared memory, thread (j-group of 4, k-group of 4) keeps a 4x4 block of the 256 x 16 result.
__global__ void __launch_bounds__(256, 2) head_wgrad_kernel(HeadParams p, float* __restrict__ wpartial) {
  __shared__ __align__(16) float y_s[HWG_ROWS][TC_H];
  __shared__ __align__(16) float dp_s[HWG_ROWS][TC_OPAD];
  __shared__ __align__(16) float bn_s[2][TC_H];
  const int tid = threadIdx.x;
  for (int j = tid; j < TC_H; j += 256) {
    const float iv = 1.0f / sqrtf(p.var[j] + p.eps);
    bn_s[0][j] = p.gamma[j] * iv;
    bn_s[1][j] = p.beta[j] - p.gamma[j] * p.mean[j] * iv;
  }
  const int jg = tid >> 2, kg = tid & 3;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  const long rows = (long)p.B * p.T;
  const int nq = TC_H / 4;
  __syncthreads();
  for (long r0 = (long)blockIdx.x * HWG_ROWS; r0 < rows; r0 += (long)gridDim.x * HWG_ROWS) {
    // stage: 32 rows x 256 cols, each thread converts 4 x (8 bf16)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + 256 * i;            // 0..1023 = 32 rows x 32 chunks of 8
      const int rr = idx >> 5, ch = idx & 31;
      const long r = r0 + rr;
      float v[8];
      if (r < rows) {
        const long b = r / p.T;
        const int t = (int)(r % p.T);
        const uint4 raw = *reinterpret_cast<const uint4*>(p.xh + (b * (p.T + 1) + t + 1) * TC_XH_LD + ch * 8);
        const uint32_t hw[4] = {raw.x, raw.y, raw.z, raw.w};
        float dm[8];
        if (p.use_dropout) {
          const uint64_t qbase = ((uint64_t)(p.row0 + b) * p.T + t) * nq + ch * 2;
          dropout_quad(p.key, qbase, dm);
          dropout_quad(p.key, qbase + 1, dm + 4);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) dm[e] = 1.f;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          v[2 * e] = fmaf(bn_s[0][ch * 8 + 2 * e], bf16_lo(hw[e]), bn_s[1][ch * 8 + 2 * e]) * dm[2 * e];
          v[2 * e + 1] = fmaf(bn_s[0][ch * 8 + 2 * e + 1], bf16_hi(hw[e]), bn_s[1][ch * 8 + 2 * e + 1]) * dm[2 * e + 1];
        }
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
      }
      *reinterpret_cast<float4*>(&y_s[rr][ch * 8]) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(&y_s[rr][ch * 8 + 4]) = make_float4(v[4], v[5], v[6], v[7]);
    }
    for (int idx = tid; idx < HWG_ROWS * TC_OPAD; idx += 256) {
      const long r = r0 + idx / TC_OPAD;
      dp_s[idx / TC_OPAD][idx % TC_OPAD] = (r < rows) ? p.dpred[r * TC_OPAD + idx % TC_OPAD] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < HWG_ROWS; ++rr) {
      const float4 yv = *reinterpret_cast<const float4*>(&y_s[rr][jg * 4]);
      const float4 dv = *reinterpret_cast<const float4*>(&dp_s[rr][kg * 4]);
      const float ya[4] = {yv.x, yv.y, yv.z, yv.w};
      const float da[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(ya[a], da[b], acc[a][b]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
      wpartial[(long)blockIdx.x * HWG_PART + (jg * 4 + a) * TC_OPAD + kg * 4 + b] = acc[a][b];
}

// Sums the per-CTA head partials (stored [value][cta]: one warp per value, lanes over CTAs, fixed order) and
// scatters them into the flat gradient vector / loss tail.  wpartial is [cta][256*16].
__global__ void head_reduce_kernel(int n_cta, const float* __restrict__ partial, int n_wcta,
                                   const float* __restrict__ wpartial, int O, int B, const float* denom, float p1,
                                   float p2, int train, float* __restrict__ gWo, float* __restrict__ gbo,
                                   float* __restrict__ ggamma, float* __restrict__ gbeta, float* __restrict__ out2) {
  pdl_sync();
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;     // one warp per output value
  const int lane = threadIdx.x & 31;
  if (i < HWG_PART) {
    if (!train) return;
    const int j = i / TC_OPAD, k = i % TC_OPAD;
    double s = 0.0;
    for (int c = lane; c < n_wcta; c += 32) s += wpartial[(long)c * HWG_PART + i];
    s = warp_sum(s);
    if (lane == 0 && k < O) gWo[j * O + k] = (float)s;
    return;
  }
  const int q = i - HWG_PART;
  if (q >= HEAD_PART) return;
  double s = 0.0;
  for (int c = lane; c < n_cta; c += 32) s += partial[(long)q * n_cta + c];
  s = warp_sum(s);
  if (q < TC_H) {
    if (train && lane == 0) ggamma[q] = (float)s;
  } else if (q < 2 * TC_H) {
    if (train && lane == 0) gbeta[q - TC_H] = (float)s;
  } else if (q < 2 * TC_H + TC_OPAD) {
    const int k = q - 2 * TC_H;
    if (train && lane == 0 && k < O) gbo[k] = (float)s;
  } else if (q == 2 * TC_H + TC_OPAD) {
    // the three loss sums live in consecutive slots; this warp finishes the loss (losses.py:87-98)
    double s1 = 0.0, s2 = 0.0;
    for (int c = lane; c < n_cta; c += 32) {
      s1 += partial[(long)(q + 1) * n_cta + c];
      s2 += partial[(long)(q + 2) * n_cta + c];
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) {
      const double Bg = denom[0], Mg = denom[1];
      const double mse0 = s / Bg, mse1 = s1 / (Bg * O), mse2 = s2 / (Mg * O);
      out2[0] = (float)(p1 * mse0 + (1.0 - p1) * (p2 * mse1 + (1.0 - p2) * mse2));
      out2[1] = (float)mse0;
    }
  }
}

// tensor-core head, one thread per hidden unit j.  In: G = h^T dpred (in gWo), cs = colsum(dpred) (in gbo).
// With y = a_j h + c_j (a = gamma*inv, c = beta - gamma*mean*inv) and dy = dpred Wo^T:
//   dWo[j][k] = a_j G[j][k] + c_j cs[k]
//   dbeta_j   = sum_r dy[r][j]           = sum_k Wo[j][k] cs[k]
//   dgamma_j  = sum_r dy[r][j] xhat[r][j] = inv_j (sum_k Wo[j][k] G[j][k] - mean_j dbeta_j)
__global__ void head_fold_kernel(int O, float* __restrict__ gWo, const float* __restrict__ gbo,
                                 float* __restrict__ ggamma, float* __restrict__ gbeta, const float* __restrict__ Wo,
                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                 const float* __restrict__ mean, const float* __restrict__ var, float eps) {
  pdl_sync();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= TC_H) return;
  const float iv = 1.0f / sqrtf(var[j] + eps);
  const float a = gamma[j] * iv, c = beta[j] - gamma[j] * mean[j] * iv;
  float db = 0.f, sg = 0.f;
  for (int k = 0; k < O; ++k) {
    const float w = Wo[j * O + k], g = gWo[j * O + k], cs = gbo[k];
    db = fmaf(w, cs, db);
    sg = fmaf(w, g, sg);
    gWo[j * O + k] = fmaf(a, g, c * cs);
  }
  gbeta[j] = db;
  ggamma[j] = iv * (sg - mean[j] * db);
}

// ---------------------------------------------------------------------------------------------
// Training head beside the forward recurrence (dropout off, one tile iteration of the recurrence).  Launched as the
// programmatic dependent of lstm_fwd_tc_kernel<true>, whose CTAs all trigger it right after their own wait: the grid
// is dispatched once the whole recurrence is resident and lands on the SMs it leaves idle (the shared memory below
// cannot fit beside a forward CTA, and only one fits per SM).  CTA j owns the row tiles bt = j, j+G, .. and walks
// (t, tile) in t order; the h_t tile is fetched once the forward has counted step t on the tile's counter.  Per tile it does exactly what head_tc_kernel<true> does: pred = h WoTp + bop on tcgen05, the masked
// weighted-MSE terms, the bf16 dpred tile TMA-stored for the backward recurrence, h^T dpred accumulated in TMEM.
// Loss sums, colsum(dpred) and h^T dpred go to fixed per-CTA slots, summed in a fixed order: the results depend only
// on the inputs.  The forward never waits on this kernel.
//   warp 0: h tiles (TMA, 3-stage ring), warp 1: MMAs + dpred store, warps 2-5: one row per thread.
// ---------------------------------------------------------------------------------------------
constexpr int HP_STAGES = 3;
constexpr uint32_t HP_H = 0;                                   // HP_STAGES x 4 k-blocks x [128 x 128 B]
constexpr uint32_t HP_WOT = HP_STAGES * 65536;                 // 4 k-blocks x [16 x 128 B]
constexpr uint32_t HP_DP = HP_WOT + 8192;                      // 2 x [128 x 64 B]
constexpr uint32_t HP_BARS = HP_DP + 2 * 8192;
constexpr int HP_SMEM = HP_BARS + 256 + 1024;
constexpr int HP_THREADS = 192;
constexpr int HP_PART = 3 + TC_OPAD;                           // s0 s1 s2 | colsum(dpred), per CTA
constexpr int HP_TRACE_UNITS = 128;                            // LFMQ_TRACE_HEAD: stamps of CTA 0's first units
constexpr int SM_SMEM_BYTES = 233472;                          // shared memory per SM (228 KB)
static_assert(HP_SMEM + FWD_SMEM > SM_SMEM_BYTES, "a paced head CTA must not fit beside a forward CTA");
static_assert(2 * HP_SMEM > SM_SMEM_BYTES, "one paced head CTA per SM");

struct HpBars {
  uint64_t wt_full, w_done;
  uint64_t h_full[HP_STAGES], h_empty[HP_STAGES];
  uint64_t pred_full[2], acc_free[2], dp_full[2], dp_free[2];
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(HP_THREADS, 1)
    head_paced_kernel(HeadParams p, HeadTcWeights w, const __grid_constant__ CUtensorMap tm_h,
                      const __grid_constant__ CUtensorMap tm_wot, const __grid_constant__ CUtensorMap tm_dpb, int n_btiles,
                      int n_tiles_cap, unsigned int* __restrict__ progress, float* __restrict__ wpartial,
                      float* __restrict__ hpart) {
  // No griddepcontrol.wait before the loop: this grid runs beside the forward recurrence.  WoTp, bop, the denominators
  // and y were written by grids that the forward's own wait has already seen complete (the forward triggers this grid
  // only after that wait); h_t is acquired through progress[].  The backward may be dispatched at once: it cannot get
  // an SM before forward CTAs leave, and its own wait is on this grid, which ends only after the forward (see below).
  griddep_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  HpBars* bars = reinterpret_cast<HpBars*>(smem + HP_BARS);
  __shared__ float red_s[4][HP_PART];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int G = gridDim.x, j0 = blockIdx.x;
  const int nk = (n_btiles - j0 + G - 1) / G;       // row tiles of this CTA (G <= n_btiles, so >= 1)
  const int N = p.T * nk;                           // units (t, k), t-major
  long long* trc = (p.trace && blockIdx.x == 0) ? p.trace : nullptr;
  if (trc && tid == 0) {
    trc[0] = (long long)ld_acquire_gpu(progress + j0 * HP_CSTRIDE);   // forward steps already counted at the start
    trc[1] = (long long)globaltimer_ns();
  }
  for (int i = tid; i < 2 * 8192 / 16; i += HP_THREADS) reinterpret_cast<uint4*>(smem + HP_DP)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    mbar_init(&bars->wt_full, 1);
    mbar_init(&bars->w_done, 1);
    for (int s = 0; s < HP_STAGES; ++s) {
      mbar_init(&bars->h_full[s], 1);
      mbar_init(&bars->h_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->pred_full[a], 1);
      mbar_init(&bars->acc_free[a], 128);
      mbar_init(&bars->dp_full[a], 128);
      mbar_init(&bars->dp_free[a], 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&bars->tmem_base, 64);
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const uint32_t acc_p = tmem;             // 2 x 16 columns: pred of alternate units
  const uint32_t acc_w = tmem + 32;        // 2 x 16 columns: sum over this CTA's units of h^T dpred (rows = hidden unit)

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(&bars->wt_full, 8192);
      for (int kb = 0; kb < 4; ++kb) tma_load_2d(smem + HP_WOT + kb * 2048, &tm_wot, &bars->wt_full, kb * 64, 0);
      for (int n = 0; n < N; ++n) {
        const int t = n / nk, bt = j0 + (n % nk) * G, s = n % HP_STAGES;
        if (n >= HP_STAGES) mbar_wait(&bars->h_empty[s], ((n / HP_STAGES) - 1) & 1);
        const long long spin0 = clock64();
        while (ld_acquire_gpu(progress + bt * HP_CSTRIDE) < (unsigned int)(t + 1)) {
          // the forward is resident before this grid starts and never waits on it; should the count never come, fail
          // the launch after ~2 s instead of hanging the device
          if (clock64() - spin0 > 4000000000LL) __trap();
        }
        fence_proxy_async_global();
        if (trc && n < HP_TRACE_UNITS) trc[2 + 2 * n] = (long long)globaltimer_ns();
        mbar_arrive_expect_tx(&bars->h_full[s], 65536);
        for (int kb = 0; kb < 4; ++kb)
          tma_load_2d(smem + HP_H + s * 65536 + kb * 16384, &tm_h, &bars->h_full[s], (t + 1) * TC_XH_LD + kb * 64, bt * 128);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc_p = make_idesc_bf16(128, 16, false, false);
      const uint32_t idesc_w = make_idesc_bf16(128, 16, true, true);
      mbar_wait(&bars->wt_full, 0);
      for (int n = 0; n <= N; ++n) {
        if (n < N) {        // pred of unit n ...
          const int s = n % HP_STAGES, a = n & 1;
          mbar_wait(&bars->h_full[s], (n / HP_STAGES) & 1);
          if (n >= 2) mbar_wait(&bars->acc_free[a], ((n >> 1) - 1) & 1);
          tcgen05_fence_after();
#pragma unroll
          for (int kb = 0; kb < 4; ++kb)
#pragma unroll
            for (int k16 = 0; k16 < 4; ++k16) {
              const uint64_t da = make_smem_desc(smem_u32(smem + HP_H + s * 65536 + kb * 16384) + k16 * 32, 0, 1024,
                                                 LAYOUT_SW128);
              const uint64_t db = make_smem_desc(smem_u32(smem + HP_WOT + kb * 2048) + k16 * 32, 0, 1024, LAYOUT_SW128);
              umma_f16(acc_p + a * 16, da, db, idesc_p, (kb | k16) != 0);
            }
          umma_commit(&bars->pred_full[a]);
        }
        if (n >= 1) {       // ... while the rows finish unit n-1: its dpred tile to HBM and into h^T dpred
          const int u = n - 1, s = u % HP_STAGES, d = u & 1;
          const int t = u / nk, bt = j0 + (u % nk) * G;
          mbar_wait(&bars->dp_full[d], (u >> 1) & 1);
          tcgen05_fence_after();
          tma_store_2d(&tm_dpb, smem + HP_DP + d * 8192, 0, (t * n_tiles_cap + bt) * 128);
          bulk_commit_group();
#pragma unroll
          for (int mb = 0; mb < 2; ++mb)
#pragma unroll
            for (int k16 = 0; k16 < 8; ++k16) {
              const uint64_t wa = make_smem_desc(smem_u32(smem + HP_H + s * 65536 + 2 * mb * 16384) + k16 * 2048, 16384,
                                                 1024, LAYOUT_SW128);
              const uint64_t wb = make_smem_desc(smem_u32(smem + HP_DP + d * 8192) + k16 * 1024, 0, 512, LAYOUT_SW64);
              umma_f16(acc_w + mb * 16, wa, wb, idesc_w, (u > 0 || k16 > 0) ? 1u : 0u);
            }
          umma_commit(&bars->h_empty[s]);     // both MMAs of unit u are done with the h stage
          bulk_wait_group_read0();            // the store has read the dpred tile ...
          umma_commit(&bars->dp_free[d]);     // ... and the h^T dpred MMAs are done with it
          if (trc && u < HP_TRACE_UNITS) trc[3 + 2 * u] = (long long)globaltimer_ns();
        }
      }
      umma_commit(&bars->w_done);
      bulk_wait_group0();
    }
  } else {
    const int wq = warp & 3;                // TMEM lane quadrant of this warp
    const int mrow = wq * 32 + lane;        // row this thread can reach in TMEM == row it owns
    const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
    const float Bg = p.denom[0], Mg = p.denom[1];
    const float c_all = (1.f - p.p1) * (1.f - p.p2) / ((float)p.O * Mg);
    const float c_last = (1.f - p.p1) * p.p2 / (Bg * (float)p.O);
    const float c_tar = p.p1 / Bg;
    float bop[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) bop[k] = w.bop[k];
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    float accbo[TC_OPAD];
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) accbo[k] = 0.f;
    // y of a unit does not depend on the forward: fetched one unit ahead
    auto load_y = [&](int n, float* yv) {
      const int t = n / nk, bt = j0 + (n % nk) * G;
      const long b = (long)bt * 128 + mrow;
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) yv[k] = 0.f;
      if (b < p.B) {
        const long r = b * p.T + t;
#pragma unroll
        for (int k = 0; k < TC_OPAD; ++k)
          if (k < p.O) yv[k] = p.y[r * p.O + k];
      }
    };
    float yt[TC_OPAD];
    load_y(0, yt);
    for (int n = 0; n < N; ++n) {
      const int t = n / nk, bt = j0 + (n % nk) * G, a = n & 1;
      const bool valid = (long)bt * 128 + mrow < p.B;
      float yn[TC_OPAD];
      if (n + 1 < N) load_y(n + 1, yn);
      mbar_wait(&bars->pred_full[a], (n >> 1) & 1);
      tcgen05_fence_after();
      uint32_t pv[16];
      tmem_ld_32x32b_x16(acc_p + a * 16 + lane_addr, pv);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(&bars->acc_free[a]);
      bool any = false;
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) any |= (yt[k] != 0.0f);          // losses.py:72
      const float mk = (any && valid) ? 1.f : 0.f;
      const bool last = (t == p.T - 1);
      float dp[TC_OPAD];
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) {
        const float pr = __uint_as_float(pv[k]) + bop[k];
        const float d = (k < p.O && valid) ? (pr * mk - yt[k]) : 0.f;  // losses.py:75
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
        dp[k] = 2.f * d * coef * mk;
        accbo[k] += dp[k];
      }
      // dpred row -> [128 x 64 B] SWIZZLE_64B tile: chunk c of row m at m*64 + ((c ^ ((m>>1)&3)) << 4)
      if (n >= 2) mbar_wait(&bars->dp_free[a], ((n >> 1) - 1) & 1);
      uint8_t* drow = smem + HP_DP + a * 8192 + mrow * 64;
      const int s64 = (mrow >> 1) & 3;
      *reinterpret_cast<uint4*>(drow + ((0 ^ s64) << 4)) =
          make_uint4(pack_bf16x2(dp[0], dp[1]), pack_bf16x2(dp[2], dp[3]), pack_bf16x2(dp[4], dp[5]), pack_bf16x2(dp[6], dp[7]));
      *reinterpret_cast<uint4*>(drow + ((1 ^ s64) << 4)) =
          make_uint4(pack_bf16x2(dp[8], dp[9]), pack_bf16x2(dp[10], dp[11]), pack_bf16x2(dp[12], dp[13]), pack_bf16x2(dp[14], dp[15]));
      fence_proxy_async_smem();
      mbar_arrive(&bars->dp_full[a]);
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) yt[k] = yn[k];
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
#pragma unroll
    for (int k = 0; k < TC_OPAD; ++k) accbo[k] = warp_sum(accbo[k]);
    if (lane == 0) {
      red_s[wq][0] = s0; red_s[wq][1] = s1; red_s[wq][2] = s2;
#pragma unroll
      for (int k = 0; k < TC_OPAD; ++k) red_s[wq][3 + k] = accbo[k];
    }
    // this CTA's h^T dpred: TMEM lane = hidden unit (mod 128), 16 columns per 128-unit block
    float* wp = wpartial + (long)blockIdx.x * HWG_PART;
    mbar_wait(&bars->w_done, 0);
    tcgen05_fence_after();
#pragma unroll
    for (int mb = 0; mb < 2; ++mb) {
      uint32_t v[16];
      tmem_ld_32x32b_x16(acc_w + lane_addr + mb * 16, v);
      tmem_ld_wait();
      float* o = wp + (mb * 128 + mrow) * TC_OPAD;
#pragma unroll
      for (int k4 = 0; k4 < 16; k4 += 4)
        *reinterpret_cast<float4*>(o + k4) = make_float4(__uint_as_float(v[k4]), __uint_as_float(v[k4 + 1]),
                                                         __uint_as_float(v[k4 + 2]), __uint_as_float(v[k4 + 3]));
    }
  }
  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (tid < HP_PART) hpart[(long)blockIdx.x * HP_PART + tid] = ((red_s[0][tid] + red_s[1][tid]) + red_s[2][tid]) + red_s[3][tid];
  if (warp == 0) tmem_dealloc(tmem, 64);
  // The forward is complete past this wait, so (1) its counts on this CTA's tiles are final and can be reset for the
  // next call -- only this CTA reads them, and the next forward is ordered after this grid -- and (2) the next kernel
  // (the backward, whose wait is on this grid) sees the forward's deferred saved-state stores.
  griddep_wait();
  for (int bt = j0 + tid * G; bt < n_btiles; bt += G * HP_THREADS) progress[bt * HP_CSTRIDE] = 0u;
}

// What the paced head leaves per CTA, reduced and folded into the head gradients and the loss by the launch that also
// reduces the weight gradient (wgrad_head_reduce_kernel).
struct HeadFoldArgs {
  int G, O;
  const float* hpart;          // [G][HP_PART]
  const float* wpart;          // [G][256 * 16]  h^T dpred
  const float* denom;
  float p1, p2, eps;
  const float *Wo, *gamma, *beta, *mean, *var;
  float *gWo, *gbo, *ggamma, *gbeta, *out2;
};
constexpr int HF_UNITS = 16;                            // hidden units per fold block
constexpr int HF_BLOCKS = TC_H / HF_UNITS + 1;          // + one block for the loss

// Block bid < TC_H / HF_UNITS: sums (in double, CTA order) h^T dpred for its 16 hidden units and colsum(dpred), then
// the fold of head_fold_kernel; block TC_H / HF_UNITS: the loss of head_reduce_kernel.  256 threads.
__device__ __forceinline__ void head_fold_body(int bid, const HeadFoldArgs& a) {
  __shared__ float cs_s[TC_OPAD];
  __shared__ float g_s[HF_UNITS][TC_OPAD];
  __shared__ double l_s[3];
  const int tid = threadIdx.x;
  if (bid == TC_H / HF_UNITS) {
    if (tid < 3) {
      double s = 0.0;
      for (int c = 0; c < a.G; ++c) s += a.hpart[(long)c * HP_PART + tid];
      l_s[tid] = s;
    }
    __syncthreads();
    if (tid == 0) {
      const double Bg = a.denom[0], Mg = a.denom[1];
      const double mse0 = l_s[0] / Bg, mse1 = l_s[1] / (Bg * a.O), mse2 = l_s[2] / (Mg * a.O);
      a.out2[0] = (float)(a.p1 * mse0 + (1.0 - a.p1) * (a.p2 * mse1 + (1.0 - a.p2) * mse2));
      a.out2[1] = (float)mse0;
    }
    return;
  }
  if (tid < TC_OPAD) {
    double s = 0.0;
    for (int c = 0; c < a.G; ++c) s += a.hpart[(long)c * HP_PART + 3 + tid];
    cs_s[tid] = (float)s;
    if (bid == 0 && tid < a.O) a.gbo[tid] = (float)s;
  }
  const int jl = tid / TC_OPAD, k = tid % TC_OPAD, j0 = bid * HF_UNITS;
  {
    double s = 0.0;
    for (int c = 0; c < a.G; ++c) s += a.wpart[(long)c * HWG_PART + (j0 + jl) * TC_OPAD + k];
    g_s[jl][k] = (float)s;
  }
  __syncthreads();
  if (tid < HF_UNITS) {
    const int j = j0 + tid;
    const float iv = 1.0f / sqrtf(a.var[j] + a.eps);
    const float aa = a.gamma[j] * iv, cc = a.beta[j] - a.gamma[j] * a.mean[j] * iv;
    float db = 0.f, sg = 0.f;
    for (int q = 0; q < a.O; ++q) {
      const float wv = a.Wo[j * a.O + q], g = g_s[tid][q], cs = cs_s[q];
      db = fmaf(wv, cs, db);
      sg = fmaf(wv, g, sg);
      a.gWo[j * a.O + q] = fmaf(aa, g, cc * cs);
    }
    a.gbeta[j] = db;
    a.ggamma[j] = iv * (sg - a.mean[j] * db);
  }
}

// =============================================================================================
// Host side
// =============================================================================================
static bool tc_supported(const lfmq_config& c, char* why, size_t n) {
  if (c.rnn_cell != LFMQ_CELL_LSTM) { snprintf(why, n, "the bf16 tensor-core path is built for the LSTM cell only"); return false; }
  if (c.uq) { snprintf(why, n, "the bf16 tensor-core path is built for the point-estimate head only"); return false; }
  if (c.num_hidden != TC_H) { snprintf(why, n, "num_hidden must be 256 (got %d)", c.num_hidden); return false; }
  if (c.num_layers != 1) { snprintf(why, n, "num_layers must be 1 (got %d)", c.num_layers); return false; }
  if (c.n_inputs > 32) { snprintf(why, n, "n_inputs must be <= 32 (got %d)", c.n_inputs); return false; }
  if (c.n_outputs > TC_OPAD) { snprintf(why, n, "n_outputs must be <= 16 (got %d)", c.n_outputs); return false; }
  if (c.recurrent_dropout > 0.f) { snprintf(why, n, "recurrent_dropout is not built on the bf16 path"); return false; }
  return true;
}

bool tc_shape_supported(const lfmq_config& c) {
  char why[128];
  return tc_supported(c, why, sizeof(why));
}

void tc_layout(TcState& st, const lfmq_config& c, const TcParamOff& po, char* base, size_t& off) {
  if (c.precision != LFMQ_PREC_BF16) return;
  char why[128];
  if (!tc_supported(c, why, sizeof(why))) return;   // tc_init reports the error
  if (!st.impl) st.impl = new TcImpl;
  TcImpl& m = *st.impl;
  auto take = [&](size_t bytes) -> char* {
    char* p = base ? base + off : nullptr;
    off = (off + bytes + 1023) / 1024 * 1024;
    return p;
  };
  const size_t B = (size_t)c.max_batch, T = (size_t)c.seq_len, H = TC_H;
  m.maxB = c.max_batch; m.T = c.seq_len; m.I = c.n_inputs; m.O = c.n_outputs;
  m.eps = c.bn_epsilon;
  m.xh = reinterpret_cast<__nv_bfloat16*>(take(B * (T + 1) * TC_XH_LD * 2));
  m.Up = reinterpret_cast<__nv_bfloat16*>(take(4 * H * H * 2));
  m.Wp = reinterpret_cast<__nv_bfloat16*>(take(4 * H * 32 * 2));
  m.Ubk = reinterpret_cast<__nv_bfloat16*>(take(4 * H * H * 2));
  m.biasp = reinterpret_cast<float*>(take(4 * H * 4));
  m.WoTp = reinterpret_cast<__nv_bfloat16*>(take(TC_OPAD * H * 2));
  m.WoSp = reinterpret_cast<__nv_bfloat16*>(take(H * 32 * 2));
  m.bop = reinterpret_cast<float*>(take(TC_OPAD * 4));
  m.head_ctas = 148 * 2;
  m.head_wctas = 148 * 2;
  m.head_part_elems = (size_t)m.head_ctas * HEAD_PART;
  m.head_part = reinterpret_cast<float*>(take(m.head_part_elems * 4));
  if (!c.forward_only) {
    const size_t Bt = (B + 127) / 128 * 128;      // saved state is blocked by 128-row tiles
    m.gates = reinterpret_cast<__nv_bfloat16*>(take(Bt * T * 4 * H * 2));
    m.cst = reinterpret_cast<__nv_bfloat16*>(take(Bt * T * H * 2));
    m.dz = reinterpret_cast<__nv_bfloat16*>(take(B * (T + 1) * 4 * H * 2));
    m.dhout = reinterpret_cast<__nv_bfloat16*>(take(((B + 127) / 128 * 128) * T * H * 2));
    m.dc = nullptr;
    m.pexch = reinterpret_cast<__nv_bfloat16*>(take(((B + 127) / 128) * 2 * 16 * 128 * 64 * 2));
    m.dpred = reinterpret_cast<float*>(take(B * T * TC_OPAD * 4));
    m.dpb = reinterpret_cast<__nv_bfloat16*>(take(T * ((B + 127) / 128) * 128 * 32 * 2));
    m.head_wpart = reinterpret_cast<float*>(take((size_t)m.head_wctas * HWG_PART * 4));
    m.wg_part_elems = (size_t)64 * 384 * 1024;
    m.wg_part = reinterpret_cast<float*>(take(m.wg_part_elems * 4));
  } else {
    m.gates = nullptr; m.cst = nullptr; m.dz = nullptr; m.dhout = nullptr; m.dc = nullptr; m.wg_part = nullptr;
    m.dpred = nullptr; m.head_wpart = nullptr; m.pexch = nullptr; m.dpb = nullptr;
    m.wg_part_elems = 0;
  }
  // offsets of the tensors in the flat parameter vector: the API layer's layout() is the one place that defines them
  m.oW = po.oW; m.oU = po.oU; m.ob = po.ob; m.ogamma = po.ogamma; m.obeta = po.obeta;
  m.oWo = po.oWo; m.obo = po.obo; m.omean = po.omean; m.ovar = po.ovar;
}

int tc_init(TcState& st, const lfmq_config& c) {
  if (c.precision != LFMQ_PREC_BF16) return 0;
  char why[128];
  if (!tc_supported(c, why, sizeof(why))) {
    LFMQ_SET_ERR("LFMQ_PREC_BF16 supports the H=256 single-layer forecaster only: %s; use LFMQ_PREC_FP32", why);
    return LFMQ_ERR_UNSUPPORTED;
  }
  TcImpl& m = *st.impl;
  const size_t B = (size_t)m.maxB, T = (size_t)m.T;
  LFMQ_CUDA_CHECK(cudaMemset(m.xh, 0, B * (T + 1) * TC_XH_LD * 2));
  if (m.dz) LFMQ_CUDA_CHECK(cudaMemset(m.dz, 0, B * (T + 1) * 4 * TC_H * 2));
  const uint64_t xh_row = (uint64_t)(T + 1) * TC_XH_LD;     // elements per batch row of the 2-D view
  int rc;
  if ((rc = make_map_2d(&m.tm_h, m.xh, xh_row, B, xh_row * 2, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_2d(&m.tm_x, m.xh, xh_row, B, xh_row * 2, 32, 128, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
  if ((rc = make_map_2d(&m.tm_h128, m.xh, xh_row, B, xh_row * 2, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_2d(&m.tm_wot, m.WoTp, TC_H, TC_OPAD, TC_H * 2, 64, 16, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_2d(&m.tm_wos, m.WoSp, 32, TC_H, 64, 32, 64, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
  if (m.dpb &&
      (rc = make_map_2d(&m.tm_dpb, m.dpb, 32, (uint64_t)m.T * ((m.maxB + 127) / 128) * 128, 64, 32, 128,
                        CU_TENSOR_MAP_SWIZZLE_64B)))
    return rc;
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(head_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HT_SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(head_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, HT_SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(head_paced_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HP_SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(head_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HROWS_SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(head_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, HROWS_SMEM));
  if ((rc = make_map_2d(&m.tm_u, m.Up, TC_H, 4 * TC_H, TC_H * 2, 64, 256, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_2d(&m.tm_w, m.Wp, 32, 4 * TC_H, 64, 32, 256, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(lstm_fwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
  LFMQ_CUDA_CHECK(cudaFuncSetAttribute(lstm_fwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
  // how many 8-CTA clusters can be co-resident (one CTA per SM because of shared memory)
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(TC_NC * 37);
  cfg.blockDim = dim3(FWD_THREADS);
  cfg.dynamicSmemBytes = FWD_SMEM;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = TC_NC;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int nclusters = 0;
  LFMQ_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&nclusters, lstm_fwd_tc_kernel<true>, &cfg));
  if (nclusters < 1) {
    LFMQ_SET_ERR("no 4-CTA cluster of the forward kernel fits on this device");
    return LFMQ_ERR_UNSUPPORTED;
  }
  m.max_clusters = nclusters;
  int dev = 0;
  LFMQ_CUDA_CHECK(cudaGetDevice(&dev));
  LFMQ_CUDA_CHECK(cudaDeviceGetAttribute(&m.sm_count, cudaDevAttrMultiProcessorCount, dev));
  m.fwd_head = !(getenv("LFMQ_FWD_HEAD") && atoi(getenv("LFMQ_FWD_HEAD")) == 0);
  if (m.dpb && m.fwd_head) {
    const size_t n = (size_t)((m.maxB + 127) / 128) * HP_CSTRIDE;
    LFMQ_CUDA_CHECK(cudaMalloc(&m.head_progress, n * sizeof(unsigned int)));
    LFMQ_CUDA_CHECK(cudaMemset(m.head_progress, 0, n * sizeof(unsigned int)));
  }
  m.enabled = true;
  st.weights_dirty = 1;
  return 0;
}

void tc_destroy(TcState& st) {
  if (st.impl && st.impl->side) {
    cudaStreamSynchronize(st.impl->side);
    cudaEventDestroy(st.impl->ev_fork);
    cudaEventDestroy(st.impl->ev_join);
    cudaStreamDestroy(st.impl->side);
    cudaFree(st.impl->progress);
  }
  if (st.impl && st.impl->head_progress) cudaFree(st.impl->head_progress);
  delete st.impl;
  st.impl = nullptr;
}

static int tc_pack_weights(TcState& st, const float* params, cudaStream_t s) {
  TcImpl& m = *st.impl;
  if (!st.weights_dirty) return 0;
  const int nblk = (int)(((long)4 * TC_H * TC_H + 255) / 256);
  PackArgs a;
  a.I = m.I; a.O = m.O; a.eps = m.eps;
  a.nb_w = nblk;
  a.nb_h = (TC_H * 32 + 255) / 256;
  a.nb_u = m.pexch ? nblk : 0;      // training handle: K-slices of U for the backward recurrence
  a.W = params + m.oW; a.U = params + m.oU; a.bias = params + m.ob;
  a.Wo = params + m.oWo; a.bo = params + m.obo; a.gamma = params + m.ogamma; a.beta = params + m.obeta;
  a.mean = params + m.omean; a.var = params + m.ovar;
  a.Up = m.Up; a.Wp = m.Wp; a.Ubk = m.Ubk; a.WoTp = m.WoTp; a.WoSp = m.WoSp; a.biasp = m.biasp; a.bop = m.bop;
  if (int rc = launch_pdl(pack_all_kernel, dim3(a.nb_w + a.nb_h + a.nb_u), dim3(256), 0, s, 1, a)) return rc;
  st.weights_dirty = 0;
  return 0;
}

static int tc_run_recurrence(TcState& st, const float* x, int B, bool save, unsigned int* head_progress, cudaStream_t s) {
  TcImpl& m = *st.impl;
  const long bt = (long)B * m.T * 5;
  if (int rc = launch_pdl(xh_fill_x_kernel, dim3((int)((bt + 255) / 256)), dim3(256), 0, s, 1, B, m.T, m.I, x, m.xh)) return rc;
  const int n_tiles = (B + 127) / 128;
  FwdParams p;
  p.B = B; p.T = m.T;
  p.n_clusters = n_tiles < m.max_clusters ? n_tiles : m.max_clusters;
  p.n_iters = (n_tiles + p.n_clusters - 1) / p.n_clusters;
  p.k16_x = (m.I + 15) / 16;
  p.n_tiles_cap = (m.maxB + 127) / 128;
  p.xh = m.xh;
  p.gates = save ? m.gates : nullptr;
  p.cst = save ? m.cst : nullptr;
  p.biasp = m.biasp;
  p.head_progress = head_progress;
  static long long* trace_dev = nullptr;
  static const bool want_trace = getenv("LFMQ_TRACE_FWD") != nullptr;
  if (want_trace && !trace_dev) {
    LFMQ_CUDA_CHECK(cudaMalloc(&trace_dev, 3 * 16 * 8 * sizeof(long long)));
  }
  if (want_trace) LFMQ_CUDA_CHECK(cudaMemsetAsync(trace_dev, 0, 3 * 16 * 8 * sizeof(long long), s));
  p.trace = want_trace ? trace_dev : nullptr;
  if (save) {
    if (int rc = launch_pdl(lstm_fwd_tc_kernel<true>, dim3(TC_NC * p.n_clusters), dim3(FWD_THREADS), FWD_SMEM, s, TC_NC, p,
                            m.tm_h, m.tm_x, m.tm_u, m.tm_w))
      return rc;
  } else {
    if (int rc = launch_pdl(lstm_fwd_tc_kernel<false>, dim3(TC_NC * p.n_clusters), dim3(FWD_THREADS), FWD_SMEM, s, TC_NC, p,
                            m.tm_h, m.tm_x, m.tm_u, m.tm_w))
      return rc;
  }
  if (want_trace) {
    long long h[3 * 16 * 8];
    LFMQ_CUDA_CHECK(cudaStreamSynchronize(s));
    LFMQ_CUDA_CHECK(cudaMemcpy(h, trace_dev, sizeof(h), cudaMemcpyDeviceToHost));
    const long long t0 = h[(1 * 16 + 0) * 8 + 0];
    const char* names[3] = {"producer", "mma", "epilogue"};
    for (int t = 0; t < 16; ++t) {
      fprintf(stderr, "[trace t=%2d]", 3 * t);
      for (int r = 0; r < 3; ++r) {
        fprintf(stderr, "  %s:", names[r]);
        for (int k = 0; k < 6; ++k) {
          const long long v = h[(r * 16 + t) * 8 + k];
          fprintf(stderr, " %lld", v ? v - t0 : -1LL);
        }
      }
      fprintf(stderr, "\n");
    }
  }
  return 0;
}

static int tc_run_head(TcState& st, const lfmq_config& c, const float* params, float* grads, const float* y, int B,
                       int64_t row0, int64_t step, const float* denom, float* preds, float* out2, bool train,
                       cudaStream_t s) {
  TcImpl& m = *st.impl;
  HeadParams h;
  h.B = B; h.T = m.T; h.O = m.O; h.target_idx = c.target_idx; h.train = train ? 1 : 0;
  h.xh = m.xh;
  h.gamma = params + m.ogamma; h.beta = params + m.obeta; h.mean = params + m.omean; h.var = params + m.ovar;
  h.eps = c.bn_epsilon;
  h.Wo = params + m.oWo; h.bo = params + m.obo;
  h.y = y; h.denom = denom; h.p1 = c.target_lambda; h.p2 = c.rnn_lambda;
  h.use_dropout = (c.train && c.dropout > 0.f) ? 1 : 0;
  static long long* htrace = nullptr;
  static const bool want_htrace = getenv("LFMQ_TRACE_HEAD") != nullptr;
  if (want_htrace && !htrace) LFMQ_CUDA_CHECK(cudaMalloc(&htrace, 2 * 8 * 8 * sizeof(long long)));
  if (want_htrace) LFMQ_CUDA_CHECK(cudaMemsetAsync(htrace, 0, 2 * 8 * 8 * sizeof(long long), s));
  h.trace = want_htrace ? htrace : nullptr;
  h.key.k0 = (uint32_t)(c.seed & 0xffffffffu);
  h.key.k1 = (uint32_t)(c.seed >> 32);
  h.key.stream = 0;
  h.key.step = (uint32_t)(step & 0xffffffff);
  h.key.thr = (uint32_t)((double)c.dropout * 16777216.0);
  h.key.scale = 1.0f / (1.0f - c.dropout);
  h.row0 = row0;
  h.preds = preds;
  // dhout / fp32 dpred are only produced on the dropout (SIMT) path; the tensor-core head leaves bf16 dpred tiles (dpb)
  const bool simt_train = train && c.train && c.dropout > 0.f;
  h.dhout = simt_train ? m.dhout : nullptr;
  h.dpred = simt_train ? m.dpred : nullptr;
  h.partial = m.head_part;
  const int n_btiles = (B + 127) / 128;
  const int n_tiles_cap = (m.maxB + 127) / 128;
  int grid = m.T * n_btiles;
  if (grid > m.head_ctas) grid = m.head_ctas;
  h.partial = m.head_part;
  HeadTcWeights hw;
  hw.WoTp = m.WoTp; hw.bop = m.bop;
  const bool use_tc = !h.use_dropout;       // the BN fold into the head weights needs y = a*h + b
  int n_wcta = m.head_wctas;
  if (train) {
    if (use_tc) {
      if (int rc = launch_pdl(head_tc_kernel<true>, dim3(grid), dim3(HT_THREADS), HT_SMEM, s, 1, h, hw, m.tm_h128, m.tm_wot,
                              m.tm_dpb, n_btiles, n_tiles_cap, m.head_wpart))
        return rc;
      n_wcta = grid;
      if (want_htrace) {
        long long hh[2 * 8 * 8];
        LFMQ_CUDA_CHECK(cudaStreamSynchronize(s));
        LFMQ_CUDA_CHECK(cudaMemcpy(hh, htrace, sizeof(hh), cudaMemcpyDeviceToHost));
        const long long t0 = hh[0];
        for (int k = 0; k < 8; ++k) {
          fprintf(stderr, "[htrace tile %d]  ctl:", k);
          for (int q = 0; q < 4; ++q) fprintf(stderr, " %lld", hh[(0 * 8 + k) * 8 + q] ? hh[(0 * 8 + k) * 8 + q] - t0 : -1LL);
          fprintf(stderr, "  row:");
          for (int q = 0; q < 6; ++q) fprintf(stderr, " %lld", hh[(1 * 8 + k) * 8 + q] ? hh[(1 * 8 + k) * 8 + q] - t0 : -1LL);
          fprintf(stderr, "\n");
        }
      }
    } else {
      head_rows_kernel<true><<<grid, 128, HROWS_SMEM, s>>>(h, m.tm_h128, n_btiles, n_tiles_cap);
      LFMQ_LAUNCH_CHECK();
      head_wgrad_kernel<<<m.head_wctas, 256, 0, s>>>(h, m.head_wpart);
      LFMQ_LAUNCH_CHECK();
    }
  } else {
    if (use_tc) {
      if (int rc = launch_pdl(head_tc_kernel<false>, dim3(grid), dim3(HT_THREADS), HT_SMEM, s, 1, h, hw, m.tm_h128,
                              m.tm_wot, m.tm_wot, n_btiles, n_tiles_cap, (float*)nullptr))
        return rc;
    } else {
      head_rows_kernel<false><<<grid, 128, HROWS_SMEM, s>>>(h, m.tm_h128, n_btiles, n_tiles_cap);
      LFMQ_LAUNCH_CHECK();
    }
  }
  if (y) {
    const int n_out = HWG_PART + HEAD_PART;
    if (int rc = launch_pdl(head_reduce_kernel, dim3((n_out * 32 + 255) / 256), dim3(256), 0, s, 1, grid,
                            (const float*)m.head_part, n_wcta, (const float*)m.head_wpart, m.O, B, denom, c.target_lambda,
                            c.rnn_lambda, train ? 1 : 0, grads ? grads + m.oWo : (float*)nullptr,
                            grads ? grads + m.obo : (float*)nullptr, grads ? grads + m.ogamma : (float*)nullptr,
                            grads ? grads + m.obeta : (float*)nullptr, out2))
      return rc;
    if (train && use_tc) {
      if (int rc = launch_pdl(head_fold_kernel, dim3((TC_H + 127) / 128), dim3(128), 0, s, 1, m.O, grads + m.oWo,
                              (const float*)(grads + m.obo), grads + m.ogamma, grads + m.obeta, params + m.oWo,
                              params + m.ogamma, params + m.obeta, params + m.omean, params + m.ovar, c.bn_epsilon))
        return rc;
    }
  }
  return 0;
}

int tc_forward(TcState& st, const lfmq_config& c, const float* params, const float* x, int B, int64_t row0,
               int64_t step, float* preds, bool save, cudaStream_t s) {
  if (!st.impl || !st.impl->enabled) {
    LFMQ_SET_ERR("bf16 path not initialised");
    return LFMQ_ERR_UNSUPPORTED;
  }
  int rc;
  if ((rc = tc_pack_weights(st, params, s))) return rc;
  st.prof->begin(LFMQ_REGION_FWD, s);
  if ((rc = tc_run_recurrence(st, x, B, save, nullptr, s))) return rc;
  st.prof->end(LFMQ_REGION_FWD, s);
  if (preds) {
    st.prof->begin(LFMQ_REGION_HEAD, s);
    if ((rc = tc_run_head(st, c, params, nullptr, nullptr, B, row0, step, nullptr, preds, nullptr, false, s))) return rc;
    st.prof->end(LFMQ_REGION_HEAD, s);
  }
  return 0;
}

int tc_backward_impl(TcState& st, const lfmq_config& c, const float* params, float* grads, int B, bool fused,
                     const HeadFoldArgs* hf, cudaStream_t s);

int tc_backward(TcState& st, const lfmq_config& c, const float* params, float* grads, const float* x, const float* y,
                int B, int64_t row0, int64_t step, const float* denom, float* tail, cudaStream_t s) {
  if (!st.impl || !st.impl->enabled) {
    LFMQ_SET_ERR("bf16 path not initialised");
    return LFMQ_ERR_UNSUPPORTED;
  }
  TcImpl& m = *st.impl;
  int rc;
  if ((rc = tc_pack_weights(st, params, s))) return rc;
  const bool dropout = c.train && c.dropout > 0.f;
  // The head runs beside the forward recurrence on the SMs it leaves idle when: the tensor-core head (no dropout), one
  // tile iteration of the recurrence (every cluster resident, so the head cannot take a forward cluster's SMs), enough
  // idle SMs, and programmatic dependent launch (what dispatches the head only once the recurrence is resident).
  const int n_tiles = (B + 127) / 128;
  const int idle = m.sm_count - TC_NC * n_tiles;
  const bool paced = m.head_progress && !dropout && n_tiles <= m.max_clusters && idle >= 8 && pdl_on();
  static long long* ptrace = nullptr;
  static const bool want_ptrace = getenv("LFMQ_TRACE_HEAD") != nullptr;
  if (paced && want_ptrace) {
    const size_t ntr = 2 + 2 * HP_TRACE_UNITS;
    if (!ptrace) LFMQ_CUDA_CHECK(cudaMalloc(&ptrace, ntr * sizeof(long long)));
    LFMQ_CUDA_CHECK(cudaMemsetAsync(ptrace, 0, ntr * sizeof(long long), s));
  }
  st.prof->begin(LFMQ_REGION_FWD, s);
  if ((rc = tc_run_recurrence(st, x, B, true, paced ? m.head_progress : nullptr, s))) return rc;
  HeadFoldArgs hf;
  if (paced) {
    // nothing between the two launches (no event, no copy): the head must be dispatched while the recurrence runs
    const int G = idle < n_tiles ? idle : n_tiles;
    HeadParams h = {};
    h.B = B; h.T = m.T; h.O = m.O; h.target_idx = c.target_idx; h.train = 1;
    h.y = y; h.denom = denom; h.p1 = c.target_lambda; h.p2 = c.rnn_lambda;
    h.trace = want_ptrace ? ptrace : nullptr;
    HeadTcWeights hw;
    hw.WoTp = m.WoTp; hw.bop = m.bop;
    if ((rc = launch_pdl(head_paced_kernel, dim3(G), dim3(HP_THREADS), HP_SMEM, s, 1, h, hw, m.tm_h128, m.tm_wot, m.tm_dpb,
                         n_tiles, (m.maxB + 127) / 128, m.head_progress, m.head_wpart, m.head_part)))
      return rc;
    st.prof->end(LFMQ_REGION_FWD, s);
    if (want_ptrace) {
      // CTA 0: forward CTA-steps counted on its first tile when it started, then per unit (t, tile) the global-timer
      // time at which h_t was there and at which the unit was finished, relative to the first
      long long tr[2 + 2 * HP_TRACE_UNITS];
      LFMQ_CUDA_CHECK(cudaStreamSynchronize(s));
      LFMQ_CUDA_CHECK(cudaMemcpy(tr, ptrace, sizeof(tr), cudaMemcpyDeviceToHost));
      const int nk = (n_tiles + G - 1) / G, nu = m.T * nk < HP_TRACE_UNITS ? m.T * nk : HP_TRACE_UNITS;
      const long long t0 = tr[2];
      fprintf(stderr, "[ptrace] G=%d units/CTA0=%d forward counts at start=%lld start=%lld ns\n", G, m.T * nk, tr[0],
              tr[1] - t0);
      for (int u = 0; u < nu; ++u)
        fprintf(stderr, "[ptrace] unit %3d t=%2d ready %8lld done %8lld lag %6lld ns\n", u, u / nk, tr[2 + 2 * u] - t0,
                tr[3 + 2 * u] - t0, tr[3 + 2 * u] - tr[2 + 2 * u]);
    }
    hf.G = G; hf.O = m.O;
    hf.hpart = m.head_part; hf.wpart = m.head_wpart;
    hf.denom = denom; hf.p1 = c.target_lambda; hf.p2 = c.rnn_lambda; hf.eps = c.bn_epsilon;
    hf.Wo = params + m.oWo; hf.gamma = params + m.ogamma; hf.beta = params + m.obeta; hf.mean = params + m.omean;
    hf.var = params + m.ovar;
    hf.gWo = grads + m.oWo; hf.gbo = grads + m.obo; hf.ggamma = grads + m.ogamma; hf.gbeta = grads + m.obeta;
    hf.out2 = tail;
  } else {
    st.prof->end(LFMQ_REGION_FWD, s);
    st.prof->begin(LFMQ_REGION_HEAD, s);
    if ((rc = tc_run_head(st, c, params, grads, y, B, row0, step, denom, nullptr, tail, true, s))) return rc;
    st.prof->end(LFMQ_REGION_HEAD, s);
  }
  // the tensor-core head (no dropout) leaves dLoss/dpred tiles for the backward kernel to expand on its own MMAs
  return tc_backward_impl(st, c, params, grads, B, /*fused=*/!dropout, paced ? &hf : nullptr, s);
}

}  // namespace lfmq

// =============================================================================================
// Persistent backward recurrence (reverse t inside the kernel), clusters of 4 CTAs per 128-row tile.
//   CTA r owns hidden units [64r, 64r+64): it computes dz_t for its 256 gate columns (pointwise, SURVEY App. A.4),
//   keeps them as the A operand in shared memory and multiplies by ITS K-slice of U (resident for the whole unroll):
//       partial_r[128 x 256] = dz_t[:, own 256 gate cols] * U[all 256 hidden, own gate cols]^T       (tcgen05)
//   dh_{t-1}[:, slice q] = sum_r partial_r[:, slice q]: the three foreign 128x64 slices travel as bf16 through a
//   global scratch (written with STG.256, fetched with one 1-D bulk copy per slice) -- a reduce-scatter whose volume
//   (48 KB in per CTA and step) is 5x smaller than all-gathering dz; DSMEM would cost ~3700 cycles for it
//   (profiles/r01_tc_probe.txt).
//   K order inside the slice: k' = 64*jb + 16*g + jj  <->  gate column g*H + 64r + 16*jb + jj, so hidden chunk jb
//   (16 units x 4 gates) is one 64-wide k-block and its MMAs overlap the pointwise work of chunk jb+1.
// =============================================================================================
namespace lfmq {

struct BwdParams {
  int B, T, n_iters, n_clusters, n_tiles_cap;
  const __nv_bfloat16* gates;
  const __nv_bfloat16* cst;
  const __nv_bfloat16* dhout;
  __nv_bfloat16* dz;
  __nv_bfloat16* pexch;      // [tile][parity][src][dst][16-column block][128][16]
  long long* trace;          // debug (LFMQ_TRACE_BWD=1)
  unsigned long long* progress;   // null, or where CTA 0 publishes base + (steps it has completed)
  unsigned long long base;
};

#define BWD_TRACE(role, k, pt)                                                                            \
  do {                                                                                                    \
    if (p.trace && blockIdx.x == 0 && (k) % 3 == 0) p.trace[((role) * 16 + (k) / 3) * 8 + (pt)] = clock64();      \
  } while (0)

constexpr int BWD_NC = 4;
// Partial exchange through L2: st.global of the foreign slices, a cluster arrive, one 1-D bulk copy per slice by the
// peer's producer.  The exchange scratch is [16-column block][row][16], so a warp's 256-bit export store is 1 KB
// contiguous and the receiver reads its 16 KB slice as it lands.  Rejected alternatives, measured on a B200:
//   pushing the slices into the peers' shared memory with st.async: profiles/r02_time_c19_dsmem_exchange.txt
//   a row-major scratch fetched with a 2-D TMA load: profiles/r02_time_c26_blocked_exchange.txt
//   per-warp peer signalling, next operands after the export: profiles/r02_time_c20_bwd_variants.txt
// Warp roles, by warpgroup (setmaxnreg moves registers between warpgroups): warps 0-3 pointwise set 0, warps 4-7 pointwise
// set 1, warps 8-11 = producer, MMA issuer, dz store, idle.  The role warpgroup gives its registers up (72 each), the
// pointwise warps take 216 (2 x 216 + 72 = the 504 of the 168 x 3 pool): the 168 of an even split left ~100 spilled values on the pointwise warps' path, with next to
// no L1 to catch them (226 KB of shared memory in use).
constexpr int BWD_THREADS = 384;
constexpr int BWD_W_PROD = 8, BWD_W_MMA = 9, BWD_W_STORE = 10;
constexpr uint32_t SB_U = 0;                    // 4 k-blocks x [256 x 128 B]
constexpr uint32_t SB_A = 131072;               // 2 stages x [128 x 128 B]
constexpr uint32_t SB_R = 163840;               // 3 foreign slices x [128 x 128 B]
constexpr uint32_t SB_DPB = 212992;             // FUSED: dLoss/dpred tile of one step [128 x 64 B], SW64
constexpr uint32_t SB_WOS = 221184;             // FUSED: (Wo gamma inv) rows of this CTA's 64 hidden units [64 x 64 B], SW64
constexpr uint32_t SB_BARS = 225280;
constexpr uint32_t BWD_SMEM = SB_BARS + 256 + 1024;

struct BwdBars {
  uint64_t w_full, a_full[2], a_empty[2], acc_full[2], recv_full, recv_free, exp_ready;
  uint64_t dpb_full, dpb_free;   // FUSED: the dpred tile has landed / the MMA reading it has completed
  uint32_t tmem_base;
};

// FUSED (no dropout in the head): dLoss/dh of the head is not read from HBM.  With dy = dpred Wo^T it equals
// dpred (Wo gamma inv)^T; the MMA warp adds that product for this CTA's 64 hidden units (two M128 x N64 x K16 MMAs per
// step on the 8 KB dpred tile) into the accumulator whose own slice the pointwise warps read anyway.
template <bool FUSED>
__global__ void __launch_bounds__(BWD_THREADS, 1)
    lstm_bwd_tc_kernel(BwdParams p, const __grid_constant__ CUtensorMap tm_ubk, const __grid_constant__ CUtensorMap tm_dzst,
                       const __grid_constant__ CUtensorMap tm_dpb, const __grid_constant__ CUtensorMap tm_wos) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  BwdBars* bars = reinterpret_cast<BwdBars*>(smem + SB_BARS);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int cid = blockIdx.x / BWD_NC;
  const int T = p.T;

  if (tid == 0) {
    mbar_init(&bars->w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->a_full[i], 128);
      mbar_init(&bars->a_empty[i], 2);      // the MMAs that read the stage have completed + the dz store has read it
      mbar_init(&bars->acc_full[i], 1);
    }
    mbar_init(&bars->recv_full, 1);
    mbar_init(&bars->recv_free, 1);
    mbar_init(&bars->exp_ready, BWD_NC - 1);   // one arrival per peer: its export for this CTA is in global memory
    mbar_init(&bars->dpb_full, 1);
    mbar_init(&bars->dpb_free, 1);
    fence_mbar_init();
  }
  if (warp == BWD_W_MMA) tmem_alloc(&bars->tmem_base, 512);
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem = bars->tmem_base;
  // programmatic dependent launch: the weight slices (packed at the start of the step) load under the predecessor's tail
  if (!(warp == BWD_W_PROD && lane == 0)) pdl_sync();

  if (warp >= 8) {
  // one setmaxnreg for the whole role warpgroup (it is warpgroup-collective), then the roles; not re-indented
  setmaxnreg_dec<72>();
  if (warp == BWD_W_PROD) {
    // ===================== TMA producer: weights once, then the foreign partial slices of every step =========
    // (an L2 prefetch of the saved activations two steps ahead was tried here and made the kernel 25 % slower)
    if (lane == 0) {
      mbar_arrive_expect_tx(&bars->w_full, 131072 + (FUSED ? 4096 : 0));
      for (int jb = 0; jb < 4; ++jb) tma_load_2d(smem + SB_U + jb * 32768, &tm_ubk, &bars->w_full, jb * 64, rank * 256);
      if (FUSED) tma_load_2d(smem + SB_WOS, &tm_wos, &bars->w_full, 0, rank * 64);
      pdl_sync();
    }
    uint32_t n_er = 0, n_dp = 0;
    // dpred tile of time step td into the single staging buffer, once the MMA that read the previous one is done
    auto load_dpred = [&](int tile, int td) {
      if (n_dp > 0) mbar_wait(&bars->dpb_free, (n_dp - 1) & 1);
      ++n_dp;
      mbar_arrive_expect_tx(&bars->dpb_full, 8192);
      tma_load_2d(smem + SB_DPB, &tm_dpb, &bars->dpb_full, 0, (td * p.n_tiles_cap + min(tile, p.n_tiles_cap - 1)) * 128);
    };
    for (int it = 0; it < p.n_iters; ++it) {
      const int tile = it * p.n_clusters + cid;
      if (FUSED && lane == 0) load_dpred(tile, T - 1);
      for (int t = T - 1; t >= 0; --t) {
        if (FUSED && lane == 0 && t > 0) load_dpred(tile, t - 1);      // for the MMA appended to this step
        if (lane == 0 && t <= T - 2) {   // step t consumes the partials exported after step t+1
          mbar_wait_cluster(&bars->exp_ready, (n_er) & 1);
          mbar_wait(&bars->recv_free, (n_er++) & 1);    // own epilogue is done reading the previous slices
          BWD_TRACE(0, T - 1 - t, 0);
          fence_proxy_async_global();
          mbar_arrive_expect_tx(&bars->recv_full, 3 * 16384);
          const int par = (t + 1) & 1;
          for (uint32_t d = 1; d < BWD_NC; ++d) {
            const uint32_t src = (rank + d) & 3;
            bulk_load_1d(smem + SB_R + (d - 1) * 16384,
                         p.pexch + ((((long)(tile * 2 + par) * 4 + (int)src) * 4 + (int)rank)) * 128 * 64, 16384,
                         &bars->recv_full);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == BWD_W_MMA) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, 256, false, false);
      const uint32_t idesc_dy = make_idesc_bf16(128, 64, false, false);
      mbar_wait(&bars->w_full, 0);
      uint32_t gs = 0;      // global step counter
      uint32_t n_dpu = 0;   // dpred tiles consumed
      // dpred(td) (Wo gamma inv)^T for this CTA's 64 hidden units into `dst` (own columns of an accumulator buffer)
      auto dy_mma = [&](uint32_t dst, bool accumulate) {
        mbar_wait(&bars->dpb_full, (n_dpu++) & 1);
        tcgen05_fence_after();
#pragma unroll
        for (int k16 = 0; k16 < 2; ++k16) {
          const uint64_t da = make_smem_desc(smem_u32(smem + SB_DPB) + k16 * 32, 0, 512, LAYOUT_SW64);
          const uint64_t db = make_smem_desc(smem_u32(smem + SB_WOS) + k16 * 32, 0, 512, LAYOUT_SW64);
          umma_f16(dst, da, db, idesc_dy, (accumulate || k16 > 0) ? 1u : 0u);
        }
        umma_commit(&bars->dpb_free);
      };
      for (int it = 0; it < p.n_iters; ++it) {
        if (FUSED) {        // dLoss/dh of the head for the tile's first step (t = T-1): nothing recurrent to add to yet
          const uint32_t pb = (gs + 1) & 1;
          dy_mma(tmem + pb * 256 + rank * 64, false);
          umma_commit(&bars->acc_full[pb]);
        }
        for (int t = T - 1; t >= 0; --t, ++gs) {
          const uint32_t acc = tmem + (gs & 1) * 256;
          for (int jb = 0; jb < 4; ++jb) {
            const uint32_t st = jb & 1;                      // stage = producing warp-set
            const uint32_t n_use = gs * 2 + (jb >> 1);
            mbar_wait(&bars->a_full[st], n_use & 1);
            if (jb == 0) BWD_TRACE(1, T - 1 - t, 0);
            if (jb == 3) BWD_TRACE(1, T - 1 - t, 1);
            tcgen05_fence_after();
#pragma unroll
            for (int k16 = 0; k16 < 4; ++k16) {
              const uint64_t da = make_smem_desc(smem_u32(smem + SB_A + st * 16384) + k16 * 32, 0, 1024, LAYOUT_SW128);
              const uint64_t db = make_smem_desc(smem_u32(smem + SB_U + jb * 32768) + k16 * 32, 0, 1024, LAYOUT_SW128);
              umma_f16(acc, da, db, idesc, (jb | k16) != 0);
            }
            umma_commit(&bars->a_empty[st]);
          }
          if (FUSED && t > 0) dy_mma(acc + rank * 64, true);      // head part of dLoss/dh_{t-1}, read as `rec` next step
          umma_commit(&bars->acc_full[gs & 1]);
          BWD_TRACE(1, T - 1 - t, 2);
        }
      }
    }
  } else if (warp == BWD_W_STORE) {
    // ===================== dz store warp =====================
    // dz_t of every staged chunk leaves for HBM straight from the A operand: one TMA store (128 rows x 128 B, rows >= B
    // clipped) instead of four STG.256 per pointwise thread.  dz keeps the operand's column order [16-unit block][gate][16]
    // (see tc_layout); wgrad_reduce_kernel puts the gate columns back in order.  A warp of its own: the wait for the
    // store's shared-memory read (~1.5 K cycles per chunk, profiles/r01_btrace_v6) used to sit on the MMA thread, between
    // the last chunk's MMAs and the commit the exchange waits for.
    // (Keeping two stores in flight -- issuing chunk i before waiting for chunk i-1's read -- was measured and lost:
    // 0.397 ms against 0.384 ms with the prefetch helper, 0.451 against 0.43 without, profiles/r02_summary.md.)
    if (lane == 0) {
      uint32_t gs = 0;
      for (int it = 0; it < p.n_iters; ++it) {
        for (int t = T - 1; t >= 0; --t, ++gs) {
          for (int jb = 0; jb < 4; ++jb) {
            const uint32_t st = jb & 1;
            const uint32_t n_use = gs * 2 + (jb >> 1);
            mbar_wait(&bars->a_full[st], n_use & 1);
            tma_store_3d(&tm_dzst, smem + SB_A + st * 16384, (4 * (int)rank + jb) * 64, t,
                         (it * p.n_clusters + cid) * 128);
            bulk_commit_group();
            bulk_wait_group_read0();
            mbar_arrive(&bars->a_empty[st]);
          }
        }
      }
      bulk_wait_group0();                        // all dz stores complete before the kernel ends
    }
  }
  } else {
    setmaxnreg_inc<216>();
    // ===================== pointwise gate gradients, A-operand staging, partial exchange =====================
    // Two warp-sets (A: warps 2-5, B: warps 6-9) split the four 16-unit chunks of a step: set s handles chunks
    // s and s+2 and owns A-operand stage s, so two chunks' global loads are always in flight together, and each
    // set issues the loads of its first chunk of step t-1 before the exchange of step t (they do not depend on it).
    const int set = warp >> 2;               // 0 / 1
    const int wq = warp & 3;                 // TMEM lane quadrant
    const int m = wq * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(wq * 32) << 16;
    const int sw = m & 7;
    float dc[32];
    uint32_t gs = 0, n_rf = 0;
    uint32_t caf[2] = {0, 0};                // completed phases of acc_full[b] (mirrors the MMA warp's commit sequence)
    // inputs of this set's two chunks of one step (slot ci): loaded ahead of the exchange they do not depend on
    uint32_t gi[2][8], gf[2][8], gg[2][8], go[2][8], dhp[2][8], ct[2][8], cp[2][8];
    const long tstride = (long)p.n_tiles_cap * 8 * 4 * 2 * 32 * 16;   // cst elements per time step

    auto load_chunk = [&](int ci, int tile, bool valid, int t) {
      const int jb = 2 * ci + set;
      if (valid) {
        const long wblk = (((long)t * p.n_tiles_cap + tile) * 8 + 2 * rank + (jb >> 1)) * 4 + wq;
        const int hb = jb & 1;
        const __nv_bfloat16* grow = p.gates + (wblk * 8 * 32 + lane) * 16;
        const __nv_bfloat16* crow = p.cst + ((wblk * 2 + hb) * 32 + lane) * 16;
        ld_global_v8(grow + (0 * 2 + hb) * 512, gi[ci]);
        ld_global_v8(grow + (1 * 2 + hb) * 512, gf[ci]);
        ld_global_v8(grow + (2 * 2 + hb) * 512, gg[ci]);
        ld_global_v8(grow + (3 * 2 + hb) * 512, go[ci]);
        if (!FUSED)
          ld_global_v8(p.dhout + ((((((long)t * p.n_tiles_cap + tile) * 4 + rank) * 4 + wq) * 4 + jb) * 32 + lane) * 16,
                       dhp[ci]);
        // c_t was this slot's c_{t-1} one step ago (the unroll runs backwards): only the first step of a tile loads it
        if (t == T - 1) {
          ld_global_v8(crow, ct[ci]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) ct[ci][j] = cp[ci][j];
        }
        if (t > 0) {
          ld_global_v8(crow - tstride, cp[ci]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) cp[ci][j] = 0u;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          gi[ci][j] = gf[ci][j] = gg[ci][j] = go[ci][j] = dhp[ci][j] = ct[ci][j] = cp[ci][j] = 0u;
      }
    };

    for (int it = 0; it < p.n_iters; ++it) {
      const int tile = it * p.n_clusters + cid;
      const long b = (long)tile * 128 + m;
      const bool valid = b < p.B;
#pragma unroll
      for (int j = 0; j < 32; ++j) dc[j] = 0.f;
      load_chunk(0, tile, valid, T - 1);
      if (FUSED) {                             // the head's dLoss/dh_{T-1} for the own slice is in the accumulator
        const uint32_t pb = (gs + 1) & 1;
        mbar_wait(&bars->acc_full[pb], caf[pb] & 1);
        ++caf[pb];
      }
      for (int t = T - 1; t >= 0; --t, ++gs) {
        const bool has_rec = t < T - 1;
        const uint32_t acc_prev = tmem + ((gs + 1) & 1) * 256;     // partial of step t+1 (own slice still there)
        // the second chunk's operands are requested only now and land under the first chunk's arithmetic, so that only
        // one chunk's operands (48 registers, not 96) are live across the export section below (one step ahead, or the
        // first chunk's here as well, were slower: profiles/r02_summary.md, c15/c16 and c18)
        load_chunk(1, tile, valid, t);
        if (has_rec) mbar_wait(&bars->recv_full, (n_rf++) & 1);
        if (tid == 64) BWD_TRACE(2, T - 1 - t, 0);
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int jb = 2 * ci + set;
          float rec[16];
          if (has_rec || FUSED) {
            uint32_t vr[16];
            if (!has_rec) tcgen05_fence_after();
            tmem_ld_32x32b_x16(acc_prev + lane_addr + rank * 64 + jb * 16, vr);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) rec[j] = __uint_as_float(vr[j]);
#pragma unroll
            for (int d = 0; d < 3 && has_rec; ++d) {
              const uint8_t* rs = smem + SB_R + d * 16384 + (jb * 128 + m) * 32;
#pragma unroll
              for (int h2 = 0; h2 < 2; ++h2) {
                const uint4 v = *reinterpret_cast<const uint4*>(rs + (h2 << 4));
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  rec[8 * h2 + 2 * e] += bf16_lo(w[e]);
                  rec[8 * h2 + 2 * e + 1] += bf16_hi(w[e]);
                }
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) rec[j] = 0.f;
          }
          // gate-gradient algebra in packed bf16x2 (all operands arrive packed; dz leaves packed); only the carried
          // dLoss/dc stays in fp32 registers.  SURVEY App. A.4.
          uint32_t zi[8], zf[8], zg[8], zo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const uint32_t i2 = gi[ci][e], f2 = gf[ci][e], g2 = gg[ci][e], o2 = go[ci][e];
            const uint32_t dh2 = FUSED ? pack_bf16x2(rec[2 * e], rec[2 * e + 1])
                                       : add_bf16x2(dhp[ci][e], pack_bf16x2(rec[2 * e], rec[2 * e + 1]));
            const uint32_t tc2 = tanh_bf16x2(ct[ci][e]);
            const uint32_t omtc2 = fma_bf16x2(neg_bf16x2(tc2), tc2, BF16X2_ONE);        // 1 - tanh(c)^2
            const uint32_t t1 = mul_bf16x2(mul_bf16x2(dh2, o2), omtc2);                 // dh * o * (1 - tc^2)
            const float dcn0 = dc[ci * 16 + 2 * e] + bf16_lo(t1);
            const float dcn1 = dc[ci * 16 + 2 * e + 1] + bf16_hi(t1);
            dc[ci * 16 + 2 * e] = dcn0 * bf16_lo(f2);
            dc[ci * 16 + 2 * e + 1] = dcn1 * bf16_hi(f2);
            const uint32_t dcn2 = pack_bf16x2(dcn0, dcn1);
            const uint32_t omi = fma_bf16x2(neg_bf16x2(i2), i2, i2);                    // i (1 - i)
            const uint32_t omf = fma_bf16x2(neg_bf16x2(f2), f2, f2);                    // f (1 - f)
            const uint32_t omg = fma_bf16x2(neg_bf16x2(g2), g2, BF16X2_ONE);            // 1 - g^2
            const uint32_t omo = fma_bf16x2(neg_bf16x2(o2), o2, o2);                    // o (1 - o)
            zi[e] = mul_bf16x2(dcn2, mul_bf16x2(g2, omi));
            zf[e] = mul_bf16x2(dcn2, mul_bf16x2(cp[ci][e], omf));
            zg[e] = mul_bf16x2(dcn2, mul_bf16x2(i2, omg));
            zo[e] = mul_bf16x2(mul_bf16x2(dh2, tc2), omo);
          }
          // A operand k-block jb in stage `set`: row m, chunk 2g+h holds gate g, units 8h..8h+7 (SW128 K-major)
          const uint32_t n_use = gs * 2 + ci;                 // use index of this stage
          if (n_use >= 1) mbar_wait(&bars->a_empty[set], (n_use - 1) & 1);
          uint8_t* arow = smem + SB_A + set * 16384 + m * 128;
          *reinterpret_cast<uint4*>(arow + ((0 ^ sw) << 4)) = make_uint4(zi[0], zi[1], zi[2], zi[3]);
          *reinterpret_cast<uint4*>(arow + ((1 ^ sw) << 4)) = make_uint4(zi[4], zi[5], zi[6], zi[7]);
          *reinterpret_cast<uint4*>(arow + ((2 ^ sw) << 4)) = make_uint4(zf[0], zf[1], zf[2], zf[3]);
          *reinterpret_cast<uint4*>(arow + ((3 ^ sw) << 4)) = make_uint4(zf[4], zf[5], zf[6], zf[7]);
          *reinterpret_cast<uint4*>(arow + ((4 ^ sw) << 4)) = make_uint4(zg[0], zg[1], zg[2], zg[3]);
          *reinterpret_cast<uint4*>(arow + ((5 ^ sw) << 4)) = make_uint4(zg[4], zg[5], zg[6], zg[7]);
          *reinterpret_cast<uint4*>(arow + ((6 ^ sw) << 4)) = make_uint4(zo[0], zo[1], zo[2], zo[3]);
          *reinterpret_cast<uint4*>(arow + ((7 ^ sw) << 4)) = make_uint4(zo[4], zo[5], zo[6], zo[7]);
          fence_proxy_async_smem();
          mbar_arrive(&bars->a_full[set]);
          if (tid == 64 && ci == 0) BWD_TRACE(2, T - 1 - t, 1);
          if (tid == 64 && ci == 1) BWD_TRACE(2, T - 1 - t, 2);
          if (tid == 192 && ci == 0) BWD_TRACE(0, T - 1 - t, 1);     // warp-set 1 in the producer row's free slots
          if (tid == 192 && ci == 1) BWD_TRACE(0, T - 1 - t, 2);
        }
        // inputs of the next step's first chunk: independent of the exchange below.  Placement matters because the
        // SM's memory pipe is a FIFO: issued here they delay the export slightly but land before the next step
        // starts; issued after the export they arrive too late (+9 % kernel time), issued inside the chunk loop they
        // hold up the chunk's own dz / A-operand stores (+17 %).
        if (t > 0) load_chunk(0, tile, valid, t - 1);
        // ---- export the foreign slices of partial_t (needed by the peers for step t-1) ----
        if (t > 0) {
          mbar_wait(&bars->acc_full[gs & 1], caf[gs & 1] & 1);
          if (tid == 64) BWD_TRACE(2, T - 1 - t, 3);
          tcgen05_fence_after();
          const uint32_t acc = tmem + (gs & 1) * 256 + lane_addr;
          const int par = t & 1;
          // all six 16-column pieces requested from TMEM before the first is waited for: one tcgen05.ld latency
          // instead of six (the 216-register budget of the pointwise warpgroups has room for the 96 values)
          uint32_t v[6][16];
#pragma unroll
          for (uint32_t d = 1; d < BWD_NC; ++d)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
              tmem_ld_32x32b_x16(acc + ((rank + d) & 3) * 64 + set * 32 + hh * 16, v[(d - 1) * 2 + hh]);
          tmem_ld_wait();
#pragma unroll
          for (uint32_t d = 1; d < BWD_NC; ++d) {
            const uint32_t dst = (rank + d) & 3;
            __nv_bfloat16* slice = p.pexch + (((long)(tile * 2 + par) * 4 + rank) * 4 + dst) * 128 * 64;
            __nv_bfloat16* out = slice + ((long)(set * 2) * 128 + m) * 16;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const uint32_t* vv = v[(d - 1) * 2 + hh];
              uint32_t pk[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) pk[e] = pack_bf16x2(__uint_as_float(vv[2 * e]), __uint_as_float(vv[2 * e + 1]));
              st_global_v8(out + hh * 128 * 16, pk);
            }
          }
          tcgen05_fence_before();
          if (tid == 64) BWD_TRACE(2, T - 1 - t, 4);
          // all 256 pointwise threads have read the received slices and stored their export: warp 0 frees the receive
          // buffer for the own producer and tells the three peers
          named_bar_sync(1, 256);
          if (tid == 64) BWD_TRACE(2, T - 1 - t, 5);
          if (warp == 0 && lane == 0) mbar_arrive(&bars->recv_free);
          if (warp == 0 && lane >= 1 && lane < BWD_NC) {
            mbar_arrive_cluster(mapa_u32(smem_u32(&bars->exp_ready), (rank + (uint32_t)lane) & 3));
          }
        }
        ++caf[gs & 1];                         // the MMA warp commits acc_full[gs & 1] every step, also at t = 0
        if (p.progress && blockIdx.x == 0 && tid == 64)
          *reinterpret_cast<volatile unsigned long long*>(p.progress) = p.base + (unsigned long long)(it * T + (T - t));
      }
    }
  }
  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == BWD_W_MMA) tmem_dealloc(tmem, 512);
}

// =============================================================================================
// Weight gradients as ONE tcgen05 GEMM over all B*(T+1) rows:  D[384 x 1024] = xh^T * dz   (both MN-major)
//   rows 0..255 -> dU, rows 256..256+I-1 -> dW, row 288 (the constant-one column) -> db.
// grid = (3 M-tiles, 4 N-tiles, S K-splits); deterministic split-K through fp32 partials.
// =============================================================================================
struct WgradParams {
  int n_kblocks;        // ceil(rows / 64)
  int kb_per_split;
  float* partial;       // [S][384][1024]
};

constexpr int WG_THREADS = 192;
constexpr int WG_STAGES = 4;
constexpr uint32_t WG_STAGE_BYTES = 16384 + 32768;
constexpr uint32_t WG_SMEM = WG_STAGES * WG_STAGE_BYTES + 1024 + 256;

__global__ void __launch_bounds__(WG_THREADS, 1)
    wgrad_tc_kernel(WgradParams p, const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b) {
  pdl_sync();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + WG_STAGES * WG_STAGE_BYTES);
  uint64_t* empty = full + WG_STAGES;
  uint64_t* acc_full = empty + WG_STAGES;
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 256;
  const int kb_beg = blockIdx.z * p.kb_per_split;
  const int kb_end = min(p.n_kblocks, kb_beg + p.kb_per_split);
  const int nkb = max(0, kb_end - kb_beg);

  if (tid == 0) {
    for (int s = 0; s < WG_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_base_s, 256);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % WG_STAGES;
        if (i >= WG_STAGES) mbar_wait(&empty[s], ((i / WG_STAGES) - 1) & 1);
        mbar_arrive_expect_tx(&full[s], WG_STAGE_BYTES);
        uint8_t* st = smem + s * WG_STAGE_BYTES;
        const int krow = (kb_beg + i) * 64;
        for (int mb = 0; mb < 2; ++mb) tma_load_2d(st + mb * 8192, &tm_a, &full[s], m0 + mb * 64, krow);
        for (int nb = 0; nb < 4; ++nb) tma_load_2d(st + 16384 + nb * 8192, &tm_b, &full[s], n0 + nb * 64, krow);
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {
      const uint32_t idesc = make_idesc_bf16(128, 256, true, true);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % WG_STAGES;
        mbar_wait(&full[s], (i / WG_STAGES) & 1);
        tcgen05_fence_after();
        uint8_t* st = smem + s * WG_STAGE_BYTES;
#pragma unroll
        for (int k16 = 0; k16 < 4; ++k16) {
          const uint64_t da = make_smem_desc(smem_u32(st) + k16 * 2048, 8192, 1024, LAYOUT_SW128);
          const uint64_t db = make_smem_desc(smem_u32(st + 16384) + k16 * 2048, 8192, 1024, LAYOUT_SW128);
          umma_f16(tmem, da, db, idesc, (i | k16) != 0);
        }
        umma_commit(&empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    const int q = warp & 3;
    const int m = q * 32 + lane;
    float* out = p.partial + ((long)blockIdx.z * 384 + m0 + m) * 1024 + n0;
    if (nkb > 0) {
      mbar_wait(acc_full, 0);
      tcgen05_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < 256; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem + ((uint32_t)(q * 32) << 16) + c0, v);
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
  if (warp == 1) tmem_dealloc(tmem, 256);
}

// Sums the K-split partials and scatters D rows into dU / dW / db of the flat gradient vector.  D's columns are in
// dz's order [16-unit block][gate][16]; the gradients want gate-major columns g*H + unit.
__device__ __forceinline__ void wgrad_reduce_body(int bid, int S, int I, const float* __restrict__ partial,
                                                  float* __restrict__ gU, float* __restrict__ gW, float* __restrict__ gb) {
  const long idx = (long)bid * blockDim.x + threadIdx.x;
  if (idx >= (long)384 * 1024) return;
  const int row = (int)(idx / 1024), np = (int)(idx % 1024);
  const int n = ((np % 64) / 16) * TC_H + (np / 64) * 16 + (np % 16);
  float* dst = nullptr;
  if (row < TC_H) dst = gU + (long)row * 1024 + n;
  else if (row < TC_H + I) dst = gW + (long)(row - TC_H) * 1024 + n;
  else if (row == TC_ONE) dst = gb + n;
  if (!dst) return;
  float s = 0.f;
  for (int z = 0; z < S; ++z) s += partial[(long)z * 384 * 1024 + idx];
  *dst = s;
}

constexpr int WGR_BLOCKS = (384 * 1024 + 255) / 256;

__global__ void __launch_bounds__(256) wgrad_reduce_kernel(int S, int I, const float* __restrict__ partial,
                                                           float* __restrict__ gU, float* __restrict__ gW,
                                                           float* __restrict__ gb) {
  pdl_sync();
  wgrad_reduce_body(blockIdx.x, S, I, partial, gU, gW, gb);
}

// With the paced head: blocks [0, HF_BLOCKS) reduce and fold the head's partials (head_fold_body; first, because
// their serial sums over the head CTAs take longer than a reduce block), the rest the weight gradient.  Off the path
// between the two recurrences.
__global__ void __launch_bounds__(256) wgrad_head_reduce_kernel(int S, int I, const float* __restrict__ partial,
                                                                float* __restrict__ gU, float* __restrict__ gW,
                                                                float* __restrict__ gb, HeadFoldArgs hf) {
  pdl_sync();
  if (blockIdx.x < HF_BLOCKS) head_fold_body(blockIdx.x, hf);
  else wgrad_reduce_body(blockIdx.x - HF_BLOCKS, S, I, partial, gU, gW, gb);
}

// Runs beside lstm_bwd_tc_kernel on the SMs it leaves idle: pulls the saved gates / cell states of the time step that
// is `lead` steps ahead of the recurrence into L2 (per step and tile iteration they are one contiguous range), paced by
// the step counter CTA 0 of the recurrence publishes.  All 128 CTAs of the recurrence issue their preloads at the same
// moment -- 12 MB at full HBM bandwidth, on the critical path; from L2 the same burst is ~2x shorter.  Measured
// (B=4096, T=48): lead 1 0.405 ms, lead 2 0.390 ms, lead 3 0.418 ms, lead 4 / none 0.43 ms (prefetched lines do not
// survive longer than ~2 steps of the kernel's own write traffic).  It only prefetches: no effect on results.  Waits
// are bounded (1 ms, then it gives up for good), e.g. when a profiler serialises the two kernels.
__global__ void __launch_bounds__(128) bwd_prefetch_kernel(const __nv_bfloat16* gates, const __nv_bfloat16* cst, int T,
                                                          int n_iters, int n_clusters, int n_tiles, int n_tiles_cap,
                                                          int lead, const unsigned long long* progress,
                                                          unsigned long long base) {
  const int nthr = gridDim.x * blockDim.x, gt = blockIdx.x * blockDim.x + threadIdx.x;
  const long gates_tile = 8L * 4 * 8 * 32 * 16 * 2, cst_tile = 8L * 4 * 2 * 32 * 16 * 2;   // bytes per (step, tile)
  __shared__ int give_up;
  if (threadIdx.x == 0) give_up = 0;
  __syncthreads();
  for (int it = 0; it < n_iters; ++it) {
    const int tile0 = it * n_clusters;
    const int ntile = min(n_clusters, n_tiles - tile0);
    if (ntile <= 0) break;
    for (int t = T - 1; t >= 0; --t) {
      const unsigned long long need = base + (unsigned long long)max(0, it * T + (T - 1 - t) - lead);
      if (threadIdx.x == 0) {
        int spins = 0;
        while (*reinterpret_cast<const volatile unsigned long long*>(progress) < need && spins < 10000) {
          __nanosleep(100);
          ++spins;
        }
        if (spins >= 10000) give_up = 1;
      }
      __syncthreads();
      if (give_up) return;
      const char* g = reinterpret_cast<const char*>(gates) + ((long)t * n_tiles_cap + tile0) * gates_tile;
      const char* c = reinterpret_cast<const char*>(cst) + ((long)t * n_tiles_cap + tile0) * cst_tile;
      for (long off = (long)gt * 4096; off < ntile * gates_tile; off += (long)nthr * 4096) prefetch_l2_bulk(g + off, 4096);
      for (long off = (long)gt * 4096; off < ntile * cst_tile; off += (long)nthr * 4096) prefetch_l2_bulk(c + off, 4096);
    }
  }
}

int tc_backward_impl(TcState& st, const lfmq_config& c, const float* params, float* grads, int B, bool fused,
                     const HeadFoldArgs* hf, cudaStream_t s) {
  TcImpl& m = *st.impl;
  int rc;
  if (!m.bwd_ready) {
    LFMQ_CUDA_CHECK(cudaFuncSetAttribute(lstm_bwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM));
    LFMQ_CUDA_CHECK(cudaFuncSetAttribute(lstm_bwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM));
    LFMQ_CUDA_CHECK(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM));
    if ((rc = make_map_2d(&m.tm_ubk, m.Ubk, 256, 4 * TC_H, 512, 64, 256, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    cudaLaunchConfig_t qc = {};
    qc.gridDim = dim3(BWD_NC * 37);
    qc.blockDim = dim3(BWD_THREADS);
    qc.dynamicSmemBytes = BWD_SMEM;
    cudaLaunchAttribute qa[1];
    qa[0].id = cudaLaunchAttributeClusterDimension;
    qa[0].val.clusterDim.x = BWD_NC;
    qa[0].val.clusterDim.y = 1;
    qa[0].val.clusterDim.z = 1;
    qc.attrs = qa;
    qc.numAttrs = 1;
    int ncl = 0;
    LFMQ_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&ncl, lstm_bwd_tc_kernel<true>, &qc));
    if (ncl < 1) {
      LFMQ_SET_ERR("no 4-CTA cluster of the backward kernel fits on this device");
      return LFMQ_ERR_UNSUPPORTED;
    }
    m.bwd_max_clusters = ncl;
    m.bwd_ready = true;
  }
  const size_t T = (size_t)m.T;
  st.prof->begin(LFMQ_REGION_BWD, s);
  {
    BwdParams bp;
    const int n_tiles = (B + 127) / 128;
    bp.B = B; bp.T = m.T;
    bp.n_tiles_cap = (m.maxB + 127) / 128;
    bp.n_clusters = n_tiles < m.bwd_max_clusters ? n_tiles : m.bwd_max_clusters;
    bp.n_iters = (n_tiles + bp.n_clusters - 1) / bp.n_clusters;
    bp.gates = m.gates; bp.cst = m.cst; bp.dhout = m.dhout; bp.dz = m.dz; bp.pexch = m.pexch;
    static long long* btrace = nullptr;
    static const bool want_btrace = getenv("LFMQ_TRACE_BWD") != nullptr;
    if (want_btrace && !btrace) LFMQ_CUDA_CHECK(cudaMalloc(&btrace, 3 * 16 * 8 * sizeof(long long)));
    if (want_btrace) LFMQ_CUDA_CHECK(cudaMemsetAsync(btrace, 0, 3 * 16 * 8 * sizeof(long long), s));
    bp.trace = want_btrace ? btrace : nullptr;
    static const int pf_lead = getenv("LFMQ_BWD_PREFETCH") ? atoi(getenv("LFMQ_BWD_PREFETCH")) : 2;   // 0 = off
    bp.progress = nullptr;
    bp.base = 0;
    if (pf_lead > 0) {
      if (!m.side) {
        LFMQ_CUDA_CHECK(cudaStreamCreateWithFlags(&m.side, cudaStreamNonBlocking));
        LFMQ_CUDA_CHECK(cudaEventCreateWithFlags(&m.ev_fork, cudaEventDisableTiming));
        LFMQ_CUDA_CHECK(cudaEventCreateWithFlags(&m.ev_join, cudaEventDisableTiming));
        LFMQ_CUDA_CHECK(cudaMalloc(&m.progress, sizeof(unsigned long long)));
        LFMQ_CUDA_CHECK(cudaMemset(m.progress, 0, sizeof(unsigned long long)));
      }
      bp.progress = m.progress;
      bp.base = m.epoch;
      m.epoch += (unsigned long long)T * bp.n_iters;
    }
    // dz as [b][t][1024] with columns ordered [16-unit block][gate][16]: one staged chunk = 128 rows x 64 columns
    CUtensorMap tm_dzst;
    {
      const uint64_t dims[3] = {1024, (uint64_t)(T + 1), (uint64_t)B};
      const uint64_t strides[2] = {2048, (uint64_t)2048 * (T + 1)};
      const uint32_t box[3] = {64, 1, 128};
      if ((rc = make_map_nd(&tm_dzst, m.dz, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    }
    if (pf_lead > 0) {
      LFMQ_CUDA_CHECK(cudaEventRecord(m.ev_fork, s));
      LFMQ_CUDA_CHECK(cudaStreamWaitEvent(m.side, m.ev_fork, 0));
      bwd_prefetch_kernel<<<20, 128, 0, m.side>>>(m.gates, m.cst, T, bp.n_iters, bp.n_clusters, n_tiles, bp.n_tiles_cap,
                                                  pf_lead, m.progress, bp.base);
      g_launches++;
      LFMQ_CUDA_CHECK(cudaEventRecord(m.ev_join, m.side));
    }
    if (fused) {
      if ((rc = launch_pdl(lstm_bwd_tc_kernel<true>, dim3(BWD_NC * bp.n_clusters), dim3(BWD_THREADS), BWD_SMEM, s, BWD_NC, bp,
                           m.tm_ubk, tm_dzst, m.tm_dpb, m.tm_wos)))
        return rc;
    } else {
      if ((rc = launch_pdl(lstm_bwd_tc_kernel<false>, dim3(BWD_NC * bp.n_clusters), dim3(BWD_THREADS), BWD_SMEM, s, BWD_NC, bp,
                           m.tm_ubk, tm_dzst, m.tm_dpb, m.tm_wos)))
        return rc;
    }
    if (pf_lead > 0) LFMQ_CUDA_CHECK(cudaStreamWaitEvent(s, m.ev_join, 0));
    if (want_btrace) {
      long long h[3 * 16 * 8];
      LFMQ_CUDA_CHECK(cudaStreamSynchronize(s));
      LFMQ_CUDA_CHECK(cudaMemcpy(h, btrace, sizeof(h), cudaMemcpyDeviceToHost));
      const long long t0 = h[(2 * 16 + 0) * 8 + 0];
      const char* names[3] = {"producer", "mma", "epilogue"};
      for (int k = 0; k < 16; ++k) {
        fprintf(stderr, "[btrace k=%2d]", 3 * k);
        for (int r = 0; r < 3; ++r) {
          fprintf(stderr, "  %s:", names[r]);
          for (int q = 0; q < 6; ++q) {
            const long long v = h[(r * 16 + k) * 8 + q];
            fprintf(stderr, " %lld", v ? v - t0 : -1LL);
          }
        }
        fprintf(stderr, "\n");
      }
    }
  }
  st.prof->end(LFMQ_REGION_BWD, s);

  st.prof->begin(LFMQ_REGION_WGRAD, s);
  // MN-major maps over exactly the B*(T+1) rows of this call (rows beyond are zero-filled by TMA)
  const uint64_t rows = (uint64_t)B * (T + 1);
  CUtensorMap tm_a, tm_b;
  if ((rc = make_map_2d(&tm_a, m.xh, TC_XH_LD, rows, TC_XH_LD * 2, 64, 64, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_2d(&tm_b, m.dz, 4 * TC_H, rows, 4 * TC_H * 2, 64, 64, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  WgradParams wp;
  wp.n_kblocks = (int)((rows + 63) / 64);
  int S = 12;
  if (wp.n_kblocks < S) S = wp.n_kblocks;
  wp.kb_per_split = (wp.n_kblocks + S - 1) / S;
  S = (wp.n_kblocks + wp.kb_per_split - 1) / wp.kb_per_split;
  wp.partial = m.wg_part;
  if ((rc = launch_pdl(wgrad_tc_kernel, dim3(3, 4, S), dim3(WG_THREADS), WG_SMEM, s, 1, wp, tm_a, tm_b))) return rc;
  if (hf) {
    if ((rc = launch_pdl(wgrad_head_reduce_kernel, dim3(WGR_BLOCKS + HF_BLOCKS), dim3(256), 0, s, 1, S, m.I,
                         (const float*)m.wg_part, grads + m.oU, grads + m.oW, grads + m.ob, *hf)))
      return rc;
  } else {
    if ((rc = launch_pdl(wgrad_reduce_kernel, dim3(WGR_BLOCKS), dim3(256), 0, s, 1, S, m.I, (const float*)m.wg_part,
                         grads + m.oU, grads + m.oW, grads + m.ob)))
      return rc;
  }
  st.prof->end(LFMQ_REGION_WGRAD, s);
  (void)params;
  (void)c;
  return 0;
}

}  // namespace lfmq
