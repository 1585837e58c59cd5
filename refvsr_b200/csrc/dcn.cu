// Modulated deformable 3x3 convolution (DCNv2) as EDVR's PCD alignment uses it: mmcv modulated_deform_conv2d with
// stride 1, pad 1, dilation 1, groups 1, 8 deform groups over 64 input channels (edvr_net.py:15-58, 104-130).
//
// Both kernels read the RAW conv_offset output (edvr_net.py:51-54): for deform group g and tap k = 3*ky + kx
//   dy = om[18g + 2k], dx = om[18g + 2k + 1], m = sigmoid(om[144 + 9g + k])
// (torch.chunk + torch.cat is the identity on the first 144 channels), so no chunk / cat / sigmoid pass runs in between.
// The offsets are read as fp32: a 16-bit offset map would move a sample by up to |offset| * 2^-8 px (bf16).
//
// dcn_tc_kernel - persistent tcgen05 implicit GEMM, M = 128 consecutive output pixels, N = NB (<= 64) output channels,
// K = 9 taps x 64 channels.  There is no TMA box to shift: the A operand of each tap is GATHERED.  Eight producer warps
// build it by bilinear, mask-scaled sampling - one (pixel, deform group) pair = 8 channels = one 16-byte vector - and store
// it straight into the K-major SWIZZLE_128B layout the UMMA descriptor reads (16-byte chunk j of row r at j ^ (r % 8), as
// in conv_tc.cu / conv_rb.cu), in a ring of 4 slots.  The weights (packing.pack_tc layout 1: [9 taps][NB][64]) stay
// resident in shared memory.  One MMA warp issues 4 K-steps per tap into one of two TMEM accumulators; four epilogue warps
// add the bias, apply the activation and store NHWC while the next tile accumulates.
//
// dcn_simt_kernel - the CUDA-core variant (any dtype incl. fp32; fp32 weights of packing.pack_simt): the fp32 precision
// path and the yardstick of the tensor-core kernel.
#include "common.cuh"
#include "tc_common.cuh"

namespace rv {

static constexpr int DCN_C = 64;                          // input channels
static constexpr int DCN_OM = 216;                        // conv_offset channels: 8 groups x 9 taps x (dy, dx) + 72 mask logits
static constexpr int DCN_NST = 4;                         // A-operand ring slots
static constexpr uint32_t DCN_A_BYTES = 128u * 128u;      // 128 pixel rows x 64 channels x 2 B
static constexpr int DCN_PRODUCERS = 8;                   // sampling warps
static constexpr int DCN_THREADS = (DCN_PRODUCERS + 1 + 4) * 32;   // + MMA issuer + 4 epilogue warps
static constexpr uint32_t DCN_TMEM_COLS = 128;            // two 64-column accumulators

struct DcnP {
  const void* x;
  const float* om;
  int om_cs, H, W, cout, NB, act, out_cs, fmt, vec_ok;
  const void* w;  // TC: [9][NB][64] 16-bit swizzled image; SIMT: fp32 [576][ldw]
  int ldw;
  const float* bias;
  void* out;
};

template <typename T>
__device__ __forceinline__ void load8(const T* p, float f[8]);
template <>
__device__ __forceinline__ void load8<float>(const float* p, float f[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
// 8 16-bit values in a 16-byte vector -> fp32
__device__ __forceinline__ void unpack8(const uint4& u, __half, float f[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 v = __half22float2(h[j]);
    f[2 * j] = v.x; f[2 * j + 1] = v.y;
  }
}
__device__ __forceinline__ void unpack8(const uint4& u, __nv_bfloat16, float f[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 v = __bfloat1622float2(h[j]);
    f[2 * j] = v.x; f[2 * j + 1] = v.y;
  }
}
template <>
__device__ __forceinline__ void load8<__half>(const __half* p, float f[8]) {
  unpack8(__ldg(reinterpret_cast<const uint4*>(p)), __half(), f);
}
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float f[8]) {
  unpack8(__ldg(reinterpret_cast<const uint4*>(p)), __nv_bfloat16(), f);
}

// Bilinear corners of output pixel (py, px), deform group g, tap k = 3*ky + kx: the sample sits at
// (py - 1 + ky + dy, px - 1 + kx + dx) and is scaled by m = sigmoid(logit).  mmcv's dmcn_im2col_bilinear rules: the column
// entry is 0 when h <= -1, h >= H, w <= -1 or w >= W, and a corner outside the map contributes 0.  Branch-free: a corner
// that contributes nothing gets weight 0 and the (valid) offset of pixel 0, so every caller issues its four loads
// unconditionally and a thread keeps all of its gathers in flight at once.  `ok` = false (a row past the last pixel) gives
// four zero weights.  off[] are element offsets into x (H, W, 64).
__device__ __forceinline__ void dcn_corners(const float* om, int H, int W, int py, int px, int g, int k, bool ok,
                                            uint32_t off[4], float wt[4]) {
  const float dy = om[18 * g + 2 * k], dx = om[18 * g + 2 * k + 1], z = om[144 + 9 * g + k];
  const int ky = k / 3, kx = k - 3 * (k / 3);
  const float h = (float)(py - 1 + ky) + dy, w = (float)(px - 1 + kx) + dx;
  const bool inside = ok && h > -1.f && w > -1.f && h < (float)H && w < (float)W;
  const float m = 1.f / (1.f + expf(-z));
  const float hf = floorf(h), wf = floorf(w);
  const int h0 = inside ? (int)hf : 0, w0 = inside ? (int)wf : 0;
  const float lh = h - hf, lw = w - wf, hh = 1.f - lh, hw = 1.f - lw;
  const float bw[4] = {hh * hw, hh * lw, lh * hw, lh * lw};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int yy = h0 + (c >> 1), xx = w0 + (c & 1);
    const bool valid = inside && yy >= 0 && yy < H && xx >= 0 && xx < W;
    wt[c] = valid ? bw[c] * m : 0.f;
    off[c] = (valid ? (uint32_t)(yy * W + xx) * DCN_C : 0u) + 8u * g;
  }
}

// bias + activation + store of one output pixel's accumulator row (fp32 bit patterns from TMEM)
template <typename T>
__device__ __forceinline__ void store_row(T* out, const DcnP& p, size_t pix, const uint32_t* acc_bits, const float* bias) {
  auto val = [&](int n) { return apply_act(__uint_as_float(acc_bits[n]) + bias[n], p.act); };
#pragma unroll
  for (int n0 = 0; n0 < 64; n0 += 8) {      // compile-time column indices: the accumulator row stays in registers
    if (p.vec_ok && n0 + 8 <= p.cout) {
      uint4 o;
      T* t = reinterpret_cast<T*>(&o);
#pragma unroll
      for (int j = 0; j < 8; ++j) t[j] = from_f<T>(val(n0 + j));
      *reinterpret_cast<uint4*>(out + pix * p.out_cs + n0) = o;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (n0 + j < p.cout) out[pix * p.out_cs + n0 + j] = from_f<T>(val(n0 + j));
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(DCN_THREADS, 1) dcn_tc_kernel(const DcnP p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_w, bar_a_full[DCN_NST], bar_a_empty[DCN_NST], bar_d_full[2], bar_d_empty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ float bias_s[64];

  const uint32_t raw = tc::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const uint32_t w_bytes = 9u * (uint32_t)p.NB * 128u;      // multiple of 1024 (NB % 16 == 0)
  uint8_t* smW = smem;
  uint8_t* smA = smem + w_bytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  const int npix = p.H * p.W;
  const int ntiles = (npix + 127) / 128;

  if (threadIdx.x == 0) {
    tc::mbar_init(&bar_w, 1);
    for (int i = 0; i < DCN_NST; ++i) {
      tc::mbar_init(&bar_a_full[i], DCN_PRODUCERS);
      tc::mbar_init(&bar_a_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&bar_d_full[i], 1);
      tc::mbar_init(&bar_d_empty[i], 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == DCN_PRODUCERS) tc::tmem_alloc(&tmem_base_s, DCN_TMEM_COLS);
  for (int i = threadIdx.x; i < 64; i += blockDim.x) bias_s[i] = (i < p.cout) ? p.bias[i] : 0.f;
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp_u < DCN_PRODUCERS) {
    // ===================== producers: bilinear, mask-scaled sampling -> swizzled A slots =====================
    const T* x = reinterpret_cast<const T*>(p.x);
    const int g = threadIdx.x & 7;                 // deform group = 16-byte chunk of the operand row
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int py[4], px[4];
      bool ok[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int pix = tile * 128 + (threadIdx.x >> 3) + 32 * i;
        ok[i] = pix < npix;
        py[i] = ok[i] ? pix / p.W : 0;
        px[i] = ok[i] ? pix - py[i] * p.W : 0;
      }
      for (int k = 0; k < 9; ++k, ++it) {
        const int slot = it & (DCN_NST - 1);
        const uint32_t ph = (it / DCN_NST) & 1u;
        tc::mbar_wait(&bar_a_empty[slot], ph ^ 1u);
        uint8_t* a = smA + (size_t)slot * DCN_A_BYTES;
        uint32_t off[4][4];
        float wt[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dcn_corners(p.om + ((size_t)py[i] * p.W + px[i]) * p.om_cs, p.H, p.W, py[i], px[i], g, k, ok[i], off[i], wt[i]);
        uint4 cv[4][4];                          // all 16 gathers of this thread issued before the first blend
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) cv[i][c] = __ldg(reinterpret_cast<const uint4*>(x + off[i][c]));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = (threadIdx.x >> 3) + 32 * i;
          float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float f[8];
            unpack8(cv[i][c], T(), f);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaf(wt[i][c], f[j], v[j]);
          }
          uint4 o;
          T* t = reinterpret_cast<T*>(&o);
#pragma unroll
          for (int j = 0; j < 8; ++j) t[j] = from_f<T>(v[j]);
          *reinterpret_cast<uint4*>(a + r * 128 + ((g ^ (r & 7)) << 4)) = o;
        }
        tc::fence_proxy_async();                 // generic-proxy smem writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&bar_a_full[slot]);
      }
    }
  } else if (warp_u == DCN_PRODUCERS) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = tc::umma_idesc(p.fmt, 128, p.NB);
    const uint64_t a_desc = tc::umma_desc_sw128(tc::smem_u32(smA));
    const uint64_t w_desc = tc::umma_desc_sw128(tc::smem_u32(smW));
    const uint32_t b_tap = ((uint32_t)p.NB * 128u) >> 4;
    if (tc::elect_one()) {
      tc::mbar_expect_tx(&bar_w, w_bytes);
      tc::bulk_load(p.w, &bar_w, smW, w_bytes);
    }
    __syncwarp();
    tc::mbar_wait(&bar_w, 0);
    uint32_t it = 0, t = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++t) {
      const uint32_t acc = t & 1u;
      tc::mbar_wait(&bar_d_empty[acc], ((t >> 1) & 1u) ^ 1u);
      tc::tc_fence_after();
      for (int k = 0; k < 9; ++k, ++it) {
        const int slot = it & (DCN_NST - 1);
        tc::mbar_wait(&bar_a_full[slot], (it / DCN_NST) & 1u);
        tc::tc_fence_after();
        if (tc::elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            tc::umma_f16(tmem_base + acc * 64u, a_desc + (uint64_t)(slot * (DCN_A_BYTES >> 4) + kk * 2),
                         w_desc + (uint64_t)(k * b_tap + kk * 2), idesc, (k | kk) ? 1u : 0u);
          tc::umma_commit(&bar_a_empty[slot]);   // slot free once these MMAs have read it
          if (k == 8) tc::umma_commit(&bar_d_full[acc]);
        }
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue: TMEM -> bias, activation -> NHWC =====================
    const int q = warp & 3;                        // TMEM lane quadrant this warp may read
    const int r = q * 32 + lane;
    T* out = reinterpret_cast<T*>(p.out);
    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++t) {
      const uint32_t acc = t & 1u;
      tc::mbar_wait(&bar_d_full[acc], (t >> 1) & 1u);
      tc::tc_fence_after();
      uint32_t v[64];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 64u;
      tc::tmem_ld32(taddr, v);
      tc::tmem_ld32(taddr + 32, v + 32);
      tc::tmem_ld_wait();
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bar_d_empty[acc]);
      const int pix = tile * 128 + r;
      if (pix < npix) store_row<T>(out, p, (size_t)pix, v, bias_s);
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == DCN_PRODUCERS) tc::tmem_dealloc(tmem_base, DCN_TMEM_COLS);
}

// CUDA-core variant: 64 output pixels per CTA.  Per tap, the 64 x 64 column block is sampled into shared memory (two
// (pixel, deform group) pairs per thread) next to the tap's 64 x 64 fp32 weights; then every thread accumulates 8 output
// channels of two pixels (r and r + 32) in fp32, reading both operands from shared memory.
template <typename T>
__global__ void __launch_bounds__(256) dcn_simt_kernel(const DcnP p) {
  __shared__ float col[64][DCN_C + 4];
  __shared__ __align__(16) float ws[DCN_C][64];
  const int npix = p.H * p.W;
  const int r = threadIdx.x >> 3, g = threadIdx.x & 7;   // sampling: pixel rows r, r + 32 and deform group g
  const int n0 = g * 8;                                  // accumulation: output channels n0..n0+7 of rows r, r + 32
  int pix[2], py[2], px[2];
  bool ok[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    pix[i] = blockIdx.x * 64 + r + 32 * i;
    ok[i] = pix[i] < npix;
    py[i] = ok[i] ? pix[i] / p.W : 0;
    px[i] = ok[i] ? pix[i] - py[i] * p.W : 0;
  }
  const T* x = reinterpret_cast<const T*>(p.x);
  float acc[2][8];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int k = 0; k < 9; ++k) {
    const float* wk = reinterpret_cast<const float*>(p.w) + (size_t)k * DCN_C * p.ldw;
    for (int e = threadIdx.x; e < DCN_C * 64; e += 256) {
      const int c = e >> 6, n = e & 63;
      ws[c][n] = n < p.ldw ? __ldg(wk + (size_t)c * p.ldw + n) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      uint32_t off[4];
      float wt[4], v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      dcn_corners(p.om + (ok[i] ? (size_t)pix[i] * p.om_cs : 0), p.H, p.W, py[i], px[i], g, k, ok[i], off, wt);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float f[8];
        load8<T>(x + off[c], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(wt[c], f[j], v[j]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) col[r + 32 * i][8 * g + j] = v[j];
    }
    __syncthreads();
#pragma unroll 4
    for (int c = 0; c < DCN_C; ++c) {
      const float4 w0 = *reinterpret_cast<const float4*>(&ws[c][n0]);
      const float4 w1 = *reinterpret_cast<const float4*>(&ws[c][n0 + 4]);
      const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float a = col[r + 32 * i][c];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a, wv[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  T* out = reinterpret_cast<T*>(p.out);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (!ok[i]) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (n0 + j < p.cout)
        out[(size_t)pix[i] * p.out_cs + n0 + j] = from_f<T>(apply_act(acc[i][j] + p.bias[n0 + j], p.act));
  }
}

template <typename T>
static int launch_dcn_tc(const DcnP& p, int grid, size_t smem, cudaStream_t st) {
  auto kern = dcn_tc_kernel<T>;
  static size_t configured = 0;
  if (smem > configured) {
    RV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  kern<<<grid, DCN_THREADS, smem, st>>>(p);
  RV_LAUNCH_CHECK("dcn_tc");
  return RV_OK;
}

template <typename T>
static int launch_dcn_simt(const DcnP& p, cudaStream_t st) {
  dcn_simt_kernel<T><<<cdiv((long long)p.H * p.W, 64), 256, 0, st>>>(p);
  RV_LAUNCH_CHECK("dcn_simt");
  return RV_OK;
}

}  // namespace rv

using namespace rv;

extern "C" int rv_dcn3x3(const void* x, const float* om, int om_cs, int H, int W, int dtype, const void* wpack,
                         const float* bias, int cout, int nb, int act, int impl, void* out, int out_cs, void* stream) {
  RV_REQUIRE(x && om && wpack && bias && out, "rv_dcn3x3: null argument");
  RV_REQUIRE(H > 0 && W > 0 && (long long)H * W * DCN_C < (1ll << 32), "rv_dcn3x3: bad geometry H=%d W=%d", H, W);
  RV_REQUIRE(om_cs >= DCN_OM, "rv_dcn3x3: the offset / mask map needs >= %d channels, got %d", DCN_OM, om_cs);
  RV_REQUIRE(cout > 0 && cout <= 64 && out_cs >= cout, "rv_dcn3x3: need 0 < cout <= 64 and cout <= out_cs (cout=%d out_cs=%d)",
             cout, out_cs);
  RV_REQUIRE(act >= RV_ACT_NONE && act <= RV_ACT_CLAMP3, "rv_dcn3x3: unknown activation %d", act);
  RV_REQUIRE((uintptr_t)x % 16 == 0, "rv_dcn3x3: x must be 16-byte aligned");
  DcnP p;
  p.x = x; p.om = om; p.om_cs = om_cs; p.H = H; p.W = W; p.cout = cout; p.NB = nb; p.act = act; p.out_cs = out_cs;
  p.w = wpack; p.bias = bias; p.out = out;
  p.fmt = dtype == RV_BF16 ? 1 : 0;
  p.ldw = (cout + 3) / 4 * 4;
  p.vec_ok = ((uintptr_t)out % 16 == 0) && ((out_cs * dtype_size(dtype)) % 16 == 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (impl == RV_CONV_IMPL_SIMT) {
    RV_DISPATCH_DTYPE(dtype, T, return launch_dcn_simt<T>(p, st));
  }
  RV_REQUIRE(impl == RV_CONV_IMPL_TC, "rv_dcn3x3: unknown impl %d", impl);
  RV_REQUIRE(dtype == RV_F16 || dtype == RV_BF16, "rv_dcn3x3(tc): activations must be f16/bf16");
  RV_REQUIRE(nb % 16 == 0 && nb >= cout && nb <= 64, "rv_dcn3x3(tc): nb=%d (multiple of 16, cout <= nb <= 64)", nb);
  RV_REQUIRE((uintptr_t)wpack % 16 == 0, "rv_dcn3x3(tc): wpack must be 16-byte aligned");
  static int num_sms = 0, max_smem = 0;
  if (num_sms == 0) {
    int dev = 0;
    RV_CUDA_OK(cudaGetDevice(&dev));
    RV_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    RV_CUDA_OK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  }
  const size_t smem = 1024 + 9 * (size_t)nb * 128 + DCN_NST * (size_t)DCN_A_BYTES;
  RV_REQUIRE(smem + 1024 <= (size_t)max_smem, "rv_dcn3x3(tc): %zu bytes of shared memory do not fit", smem);
  const int ntiles = (H * W + 127) / 128;
  const int grid = ntiles < num_sms ? ntiles : num_sms;
  if (dtype == RV_F16) return launch_dcn_tc<__half>(p, grid, smem, st);
  return launch_dcn_tc<__nv_bfloat16>(p, grid, smem, st);
}
