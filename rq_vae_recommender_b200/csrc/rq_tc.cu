// Tensor-core tokeniser for sm_100a: prepared codebook state + C-ABI entry points (the kernel is csrc/rq_tcx.cu).
//
// Result contract: identical to rqb200_rq_forward(mode = EVAL, ids only) -- the hard-argmin chain of
// modules/quantize.py:113-128,159-161 x L + modules/rqvae.py:125-132 (what semids.py:125 consumes).
//
// Why tensor cores: the distance term x.c^T is 2*D*K*L = 1.18 MFLOP per 3 KB item (381 FLOP/B, SURVEY 8d);
// on CUDA cores the pass is ~30x compute bound.  Why it is still exact: the fp16 product only FILTERS.
//   S_l[b,k]  = fp16(x_b) . fp16(c_{l,k})            (tcgen05.mma, fp32 accumulate in TMEM; exact power-of-two scales)
//   score_l   = cc_{l,k} - 2 (S_l - sum_{j<l} G_{jl}[id_j, k])     (G = fp32 Gram tables C_j C_l^T, so every level is
//               scored from the ONE fp16 image of x: the residual never has to be re-quantised or re-staged)
//   candidates = { k : score <= min + 4 eps_b }      eps_b bounds the fp16 rounding of the dot product (margin in the epilogue)
//   |candidates| == 1  -> that code is the exact argmin;  else the candidates are re-scored with the exact fp32
//   arithmetic of the CUDA-core kernel (sequential fp32 residual, (xx + cc) - 2 dot, first index wins ties).
//
#include "tc_common.cuh"

// csrc/rq_tcx.cu: the transposed CTA-pair kernel (codes on the TMEM lanes); shares the prepared state
// csrc/rq_tcx.cu / rq_tcx96.cu: the same kernel at two tile shapes (64 / 96 rows per CTA)
int tcx_run_r64(const float* x, int64_t ldx, int B, const void* state, int D, int L, int64_t* ids, int* stats, int sm_count,
                bool trace, cudaStream_t st);
int tcx_run_r96(const float* x, int64_t ldx, int B, const void* state, int D, int L, int64_t* ids, int* stats, int sm_count,
                bool trace, cudaStream_t st);
// TMA needs a 16-byte aligned base and row pitch; the kernel runs as CTA pairs
static int tcx_can_run(const float* x, int64_t ldx, int sm_count) {
  return ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && sm_count >= 2;
}

extern "C" int rqb200_tokenize_tc_supported(int D, int K, int L) {
  return (K == TC_K && D >= TC_KC && D <= TC_MAX_D && D % TC_KC == 0 && L >= 1 && L <= RQB_MAX_LEVELS) ? 1 : 0;
}

extern "C" size_t rqb200_tokenize_tc_state_bytes(int D, int K, int L) {
  if (!rqb200_tokenize_tc_supported(D, K, L)) return 0;
  return tc_off_blob(D, L) + (size_t)L * 2 * (D / TC_KC) * TC_BSTAGE_BYTES;
}

// ------------------------------------------------------------------------------------------------ prepare
// hcc[l][k] = cc/2 from a float64 sum (the filter's table); amax and c2max of the level
__global__ void tc_prep_stats_kernel(const float* const* cbs, int D, TcHeader* hdr, float* hcc) {
  const int l = blockIdx.y;
  const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (k >= TC_K) return;
  const float* c = cbs[l] + (int64_t)k * D;
  double s2 = 0.0;
  float mx = 0.f;
  for (int d = lane; d < D; d += 32) {
    const float v = c[d];
    s2 += (double)v * (double)v;
    mx = fmaxf(mx, fabsf(v));
  }
  s2 = warp_sum_d(s2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) {
    hcc[l * TC_K + k] = (float)(0.5 * s2);
    atomicMax(&hdr->amax_bits[l], __float_as_uint(mx));
    atomicMax(&hdr->c2_bits[l], __float_as_uint(__double2float_ru(sqrt(s2))));
  }
}

// cc[l][k] = sum_d c^2 in fp32, lane-strided fma + shuffle tree: bit-identical to rq_prep_norm_kernel (csrc/rq_simt.cu), it is
// the value the exact re-rank adds in (xx + cc) - 2 dot
__global__ void tc_prep_cc_kernel(const float* const* cbs, int D, float* cc) {
  const int l = blockIdx.y;
  const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (k >= TC_K) return;
  const float* c = cbs[l] + (int64_t)k * D;
  float s2 = 0.f;
  for (int d = lane; d < D; d += 32) s2 = fmaf(c[d], c[d], s2);
  s2 = warp_sum(s2);
  if (lane == 0) cc[l * TC_K + k] = s2;
}

__global__ void tc_prep_scale_kernel(TcHeader* hdr, int L) {
  const int l = threadIdx.x;
  if (l >= L) return;
  const float amax = __uint_as_float(hdr->amax_bits[l]);
  float sc = 1.f;
  if (amax > 0.f && isfinite(amax)) {
    int e;
    frexpf(amax, &e);          // amax = m * 2^e, m in [0.5, 1)
    e = max(-60, min(60, e));
    sc = ldexpf(1.f, -e);      // amax * sc in [0.5, 1)
  }
  hdr->lv[l].sc = sc;
}

// measured fp16 rounding of every code: chat = max_k ||c~_k||, ec = max_k ||c~_k - c_k||  (c~ = fp16(c sc) / sc), float64 sums
__global__ void tc_prep_err_kernel(const float* const* cbs, int D, TcHeader* hdr) {
  const int l = blockIdx.y;
  const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (k >= TC_K) return;
  const float sc = hdr->lv[l].sc;
  const double inv = 1.0 / (double)sc;
  const float* c = cbs[l] + (int64_t)k * D;
  double n2 = 0.0, e2 = 0.0;
  for (int d = lane; d < D; d += 32) {
    const double v = (double)c[d];
    const double t = (double)__half2float(__float2half_rn(c[d] * sc)) * inv;
    n2 += t * t;
    e2 += (t - v) * (t - v);
  }
  n2 = warp_sum_d(n2); e2 = warp_sum_d(e2);
  if (lane == 0) {   // non-negative floats order like their bit patterns; inf / NaN sort above every finite value
    atomicMax(&hdr->chat_bits[l], __float_as_uint(__double2float_ru(sqrt(n2))));
    atomicMax(&hdr->ec_bits[l], __float_as_uint(__double2float_ru(sqrt(e2))));
  }
}

__global__ void tc_prep_consts_kernel(TcHeader* hdr, int L) {
  const int l = threadIdx.x;
  if (l >= L) return;
  TcLevelConst& c = hdr->lv[l];
  c.chat = TC_INFL * __uint_as_float(hdr->chat_bits[l]);
  c.ec = TC_INFL * __uint_as_float(hdr->ec_bits[l]);
  c.c2max = __uint_as_float(hdr->c2_bits[l]);
  float g = 0.f;
  for (int j = 0; j < l; ++j) g += __uint_as_float(hdr->c2_bits[j]);
  c.prior = g;
  c.gerr = 2.38418579e-7f * (c.c2max * g + 0.5f * c.c2max * c.c2max);   // 2^-22: tables from float64 rounded once, <= 4 fp32 roundings after
}

// Bblob[(l*2+h)*nkc + kc] = 16 KB smem image of codes [128h, 128h+128) x k [64kc, 64kc+64):
// K-major, 128 B per code row, 16-byte chunks XOR-swizzled with (row & 7)  (UMMA SWIZZLE_128B canonical layout)
__global__ void tc_prep_blob_kernel(const float* const* cbs, int D, const TcHeader* hdr, __half* blob) {
  const int nkc = D / TC_KC;
  const int blk = blockIdx.x;  // (l*2+h)*nkc + kc
  const int kc = blk % nkc, h = (blk / nkc) & 1, l = blk / (2 * nkc);
  const float sc = hdr->lv[l].sc;
  const float* c = cbs[l];
  __half* out = blob + (size_t)blk * (TC_BSTAGE_BYTES / 2);
  for (int i = threadIdx.x; i < 128 * TC_KC; i += blockDim.x) {
    const int n = i / TC_KC, k = i % TC_KC;
    const float v = c[(int64_t)(h * 128 + n) * D + kc * TC_KC + k] * sc;
    const int chunk = (k >> 3) ^ (n & 7);
    out[n * 64 + chunk * 8 + (k & 7)] = __float2half_rn(v);
  }
}

// Gram table G_{j,l}[i][k] = c_{j,i} . c_{l,k} accumulated in float64 and rounded to fp32 ONCE; for j = 0 the level's cc_l[k] / 2 is
// folded in before the rounding, so the epilogue scores with one table sum:  h[k] = T[k] - S[k] / sc,
// T = cc/2 + sum_j G_{j,l}[id_j]  (argmin-equivalent to quantize.py:113-117).  16 x 16 outputs per block, k tiles of 16 through smem.
__global__ void __launch_bounds__(256) tc_prep_gram_kernel(const float* __restrict__ cj, const float* __restrict__ cl, int D,
                                                           float* __restrict__ g, int fold_cc) {
  __shared__ float sa[16][17], sb[16][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i = blockIdx.y * 16 + ty, k = blockIdx.x * 16 + tx;
  double acc = 0.0, cck = 0.0;
  for (int d0 = 0; d0 < D; d0 += 16) {
    sa[ty][tx] = cj[(int64_t)(blockIdx.y * 16 + ty) * D + d0 + tx];
    sb[ty][tx] = cl[(int64_t)(blockIdx.x * 16 + ty) * D + d0 + tx];
    __syncthreads();
#pragma unroll
    for (int d = 0; d < 16; ++d) {
      const double b = (double)sb[tx][d];
      acc += (double)sa[ty][d] * b;
      cck += b * b;
    }
    __syncthreads();
  }
  g[(size_t)i * TC_K + k] = (float)(fold_cc ? acc + 0.5 * cck : acc);
}

extern "C" int rqb200_tokenize_tc_prepare(const float* const* codebooks, int D, int K, int L, void* state,
                                          size_t state_bytes, void* stream) {
  if (!rqb200_tokenize_tc_supported(D, K, L)) {
    rqb_set_error("tokenize_tc: shape D=%d K=%d L=%d not supported (need K=256, D %% 64 == 0, 64 <= D <= 768)", D, K, L);
    return RQB_ERR_UNSUPPORTED;
  }
  RQB_CHECK_ARG(codebooks && state, "tokenize_tc_prepare: null pointer");
  if (state_bytes < rqb200_tokenize_tc_state_bytes(D, K, L)) {
    rqb_set_error("tokenize_tc_prepare: state too small");
    return RQB_ERR_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* base = reinterpret_cast<char*>(state);
  TcHeader* hdr = reinterpret_cast<TcHeader*>(base);
  float* cc = reinterpret_cast<float*>(base + tc_off_cc(L));
  float* hcc = reinterpret_cast<float*>(base + tc_off_hcc(L));
  float* gram = reinterpret_cast<float*>(base + tc_off_gram(L));
  const float** cbptr = reinterpret_cast<const float**>(base + tc_off_cbptr(L));
  __half* blob = reinterpret_cast<__half*>(base + tc_off_blob(D, L));
  float* cbf = reinterpret_cast<float*>(base + tc_off_cbf(L));
  RQB_CUDA(cudaMemsetAsync(hdr, 0, sizeof(TcHeader), st));
  // fp32 copy for the exact re-rank: 256-byte aligned rows whatever the caller's tensors look like, and the prepared state
  // no longer references caller memory after this call returns (stream order); every prepare kernel reads the copy
  const float* cbfp[RQB_MAX_LEVELS] = {};
  for (int l = 0; l < L; ++l) {
    RQB_CUDA(cudaMemcpyAsync(cbf + (size_t)l * TC_K * D, codebooks[l], sizeof(float) * TC_K * D, cudaMemcpyDeviceToDevice, st));
    cbfp[l] = cbf + (size_t)l * TC_K * D;
  }
  RQB_CUDA(cudaMemcpyAsync(cbptr, cbfp, sizeof(float*) * L, cudaMemcpyHostToDevice, st));   // pageable source: staged before the call returns
  tc_prep_stats_kernel<<<dim3(TC_K / 8, L), 256, 0, st>>>(cbptr, D, hdr, hcc);
  RQB_LAUNCH_CHECK();
  tc_prep_cc_kernel<<<dim3(TC_K / 8, L), 256, 0, st>>>(cbptr, D, cc);
  RQB_LAUNCH_CHECK();
  tc_prep_scale_kernel<<<1, 32, 0, st>>>(hdr, L);
  RQB_LAUNCH_CHECK();
  tc_prep_err_kernel<<<dim3(TC_K / 8, L), 256, 0, st>>>(cbptr, D, hdr);
  RQB_LAUNCH_CHECK();
  tc_prep_consts_kernel<<<1, 32, 0, st>>>(hdr, L);
  RQB_LAUNCH_CHECK();
  tc_prep_blob_kernel<<<L * 2 * (D / TC_KC), 256, 0, st>>>(cbptr, D, hdr, blob);
  RQB_LAUNCH_CHECK();
  for (int l = 1; l < L; ++l)
    for (int j = 0; j < l; ++j) {
      float* g = gram + (size_t)(l * (l - 1) / 2 + j) * TC_K * TC_K;
      tc_prep_gram_kernel<<<dim3(TC_K / 16, TC_K / 16), 256, 0, st>>>(cbf + (size_t)j * TC_K * D, cbf + (size_t)l * TC_K * D, D, g, j == 0);
      RQB_LAUNCH_CHECK();
    }
  return RQB_OK;
}


extern "C" int rqb200_tokenize_tc_run(const float* x, int64_t ldx, int B, const void* state, int D, int K, int L,
                                      int64_t* ids, int* stats, void* stream) {
  if (!rqb200_tokenize_tc_supported(D, K, L)) {
    rqb_set_error("tokenize_tc: shape D=%d K=%d L=%d not supported", D, K, L);
    return RQB_ERR_UNSUPPORTED;
  }
  RQB_CHECK_ARG(B >= 0 && ldx >= D && ldx < (1 << 24), "tokenize_tc_run: bad shape");
  if (B == 0) return RQB_OK;
  RQB_CHECK_ARG(x && state && ids, "tokenize_tc_run: null pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int dev = 0, sm_count = 0;
  RQB_CUDA(cudaGetDevice(&dev));
  RQB_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));     // per call: the state may live on any device
  // x reaches the kernel through TMA (tensor map over [B][D] fp32): 16-byte aligned base and row pitch
  RQB_CHECK_ARG(tcx_can_run(x, ldx, sm_count),
                "tokenize_tc_run: x must be 16-byte aligned with a row stride that is a multiple of 4 floats (and the device needs >= 2 SMs)");
  static const bool want_trace = []() { const char* e = getenv("RQB200_TC_TRACE"); return e && e[0] == '1'; }();
  const bool trace = want_trace && stats;       // tracing: the caller passes >= 4096 ints (tools/tc_native_check.cu)
  // Tile shape: 96-row CTAs move a third fewer codebook bytes and hand-offs per row and win once every CTA pair has several
  // tiles (12 101 rows: 0.041 vs 0.052 ms; 84 000: 0.193 vs 0.204); 64-row CTAs have the shorter pipeline and win below that
  // (5 000 x 256: 0.053 vs 0.072 ms).  Both return identical ids (tests/test_gpu_tc_variants.py).
  static const int force = []() { const char* e = getenv("RQB200_TC_ROWS"); return e ? atoi(e) : 0; }();
  const bool big = force ? force == 96 : (int64_t)B > 128ll * (sm_count / 2);     // more than one 64-row tile per CTA
  return big ? tcx_run_r96(x, ldx, B, state, D, L, ids, stats, sm_count, trace, st)
             : tcx_run_r64(x, ldx, B, state, D, L, ids, stats, sm_count, trace, st);
}
