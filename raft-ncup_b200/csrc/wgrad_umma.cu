// tcgen05 weight / bias gradient of a channel-last convolution (TF32x3), the tensor-core form of rnc_conv2d_cl_wgrad:
//   gw[tap][ci][co] += sum_p gy[p][co] * x[shift_tap(p)][ci],   gb[co] += sum_p gy[p][co]      (K = output pixels)
//
// Both tensors arrive channel-last, so K is their strided dimension.  Instead of MN-major operands, one pass per tensor
// transposes through shared memory and splits into TF32 hi/lo planes [B][C][H][Q][pitch] (hi = cvt.rna.tf32(v), lo = v - hi):
// every operand row is then 32 consecutive pixels of one channel, a K-major 128-byte row, and the 128B-swizzled TMA boxes,
// descriptors and kind::tf32 issue of conv_umma.cu apply unchanged.  The x planes hold one copy per horizontal filter offset
// kx: position (kx, j) of an input row holds input column stride*j + kx - kw/2 (zero outside the image), so the 32 input
// columns a tap pairs with the output columns [x0, x0+32) are one box at (x0, kx) for both strides, and every box starts at a
// 128-byte boundary of its row.  The vertical offset is the box's row coordinate (stride*yo + ky - kh/2); the TMA unit's
// zero fill provides the rows above / below the image, the row tail (the gy box is zero beyond Wo, so are the products) and
// the channel tails.  The gy pass also sums the bias gradient.
//
// GEMM tile: M = 128 output channels (gy planes, A) x N = BN input channels (x planes, B), K blocks of 32 pixels (one output
// row segment).  Per K step: gy_hi * [x_hi | x_lo] -> [main | corr] (one instruction of 2*BN columns) and gy_lo * x_hi -> corr.
// The tensor core truncates on every accumulate (DESIGN §3.2), so no TMEM accumulation runs over more than kKC K blocks
// (512 px, 64 MMAs per term): after each chunk the epilogue drains main + corr into fp32 registers (thread = one output
// channel, its share of the BN input channels); the accumulator pair is double-buffered so the drain overlaps the next chunk.
// Work items (co tile, ci tile, tap, K split) are spread over persistent CTAs; each item leaves through one atomicAdd per
// gradient element.
#include "umma_ptx.cuh"

namespace rnc {
namespace wgrad {

using namespace rnc::umma;

constexpr int kThreads = 320;        // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-9: epilogue (2 per lane group)
constexpr int kBM = 128;             // output channels per tile (TMEM lanes)
constexpr int kPx = 32;              // pixels per K block: one 128-byte row of TF32 words
constexpr int kKC = 16;              // K blocks per TMEM accumulation chunk (512 px); RNC_WGRAD_KC overrides (developer probe)
constexpr int kMinPer = 8;           // K blocks per split at least (an item's drain + atomics amortise over >= 256 px)
constexpr int kMaxStages = 6;
constexpr int kAPlane = kBM * 128;   // bytes of one gy plane box

struct Params {
  int Ho, nxt;                       // output rows, 32-px K blocks per output row
  int kw, ph, pw, stride;
  int cin, cout, ldw;
  int nco, nci, taps;
  long long nkb;                     // K blocks in total (B * Ho * nxt)
  long long per;                     // K blocks per split
  int kc;                            // K blocks per TMEM accumulation chunk
  int items, stages;
  float* gw;
};

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// item -> (co tile, ci tile, tap, K split); co tiles vary fastest, so the CTAs running at the same time share the K range in L2
struct Item {
  int cot, cit, tap;
  long long kb0, kb1;
};
__device__ __forceinline__ Item decode(const Params& p, int item) {
  Item it;
  int r = item;
  it.cot = r % p.nco; r /= p.nco;
  it.cit = r % p.nci; r /= p.nci;
  it.tap = r % p.taps;
  const int ks = r / p.taps;
  it.kb0 = static_cast<long long>(ks) * p.per;
  it.kb1 = it.kb0 + p.per < p.nkb ? it.kb0 + p.per : p.nkb;
  return it;
}

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_umma_kernel(const __grid_constant__ CUtensorMap mGh, const __grid_constant__ CUtensorMap mGl,
                  const __grid_constant__ CUtensorMap mXh, const __grid_constant__ CUtensorMap mXl, const Params p) {
  constexpr int kBPlane = BN * 128;
  constexpr int kStage = 2 * kAPlane + 2 * kBPlane;
  constexpr uint32_t kTmemCols = 4 * BN <= 128 ? 128 : 4 * BN <= 256 ? 256 : 512;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.stages * kStage);
  uint64_t* full = bars;
  uint64_t* empty = full + kMaxStages;
  uint64_t* acc_full = empty + kMaxStages;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (warp-uniform loop, one elected lane issues)
    int s_n = 0, p_n = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
      const Item it = decode(p, item);
      const int ky = it.tap / p.kw, kx = it.tap - ky * p.kw;
      const int co0 = it.cot * kBM, ci0 = it.cit * BN;
      for (long long kb = it.kb0; kb < it.kb1; ++kb) {
        const int s = s_n, par = p_n;
        if (++s_n == p.stages) { s_n = 0; p_n ^= 1; }
        mbar_wait(&empty[s], par ^ 1);
        const int xt = static_cast<int>(kb % p.nxt);
        const long long r = kb / p.nxt;
        const int yo = static_cast<int>(r % p.Ho), b = static_cast<int>(r / p.Ho);
        const int x0 = xt * kPx, yi = p.stride * yo + ky - p.ph;
        if (elect_one()) {
          unsigned char* st = smem + s * kStage;
          mbar_expect_tx(&full[s], kStage);
          tma_load_5d(st, &mGh, &full[s], x0, 0, yo, co0, b);
          tma_load_5d(st + kAPlane, &mGl, &full[s], x0, 0, yo, co0, b);
          tma_load_5d(st + 2 * kAPlane, &mXh, &full[s], x0, kx, yi, ci0, b);
          tma_load_5d(st + 2 * kAPlane + kBPlane, &mXl, &full[s], x0, kx, yi, ci0, b);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // instruction descriptor: D = F32 (bit 4), A / B = TF32 (2 at bits 7 and 10), both K-major, N >> 3 at 17, M >> 4 at 24
    const uint32_t fmt = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(kBM >> 4) << 24);
    const uint32_t idesc1 = fmt | (static_cast<uint32_t>(BN >> 3) << 17), idesc2 = fmt | (static_cast<uint32_t>((2 * BN) >> 3) << 17);
    const uint64_t desc0 = smem_desc_sw128(smem_u32(smem));
    int s_n = 0, p_n = 0, t = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
      const Item it = decode(p, item);
      for (long long c0 = it.kb0; c0 < it.kb1; c0 += p.kc, ++t) {
        const int buf = t & 1, use = t >> 1;
        mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
        tcgen05_fence_after();
        const uint32_t d_main = tmem_base + buf * 2 * BN, d_corr = d_main + BN;
        const long long c1 = c0 + p.kc < it.kb1 ? c0 + p.kc : it.kb1;
        for (long long kb = c0; kb < c1; ++kb) {
          const int s = s_n, par = p_n;
          if (++s_n == p.stages) { s_n = 0; p_n ^= 1; }
          mbar_wait(&full[s], par);
          tcgen05_fence_after();
          const uint64_t gh = desc0 + static_cast<uint32_t>(s * (kStage >> 4)), gl = gh + (kAPlane >> 4), xh = gh + (2 * kAPlane >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {      // 4 K steps of 8 TF32 words (32 bytes) per 128-byte row
              umma_tf32(d_main, gh + 2 * k, xh + 2 * k, idesc2, (kb == c0 && k == 0) ? 0u : 1u);   // gy_hi * [x_hi | x_lo]
              umma_tf32(d_corr, gl + 2 * k, xh + 2 * k, idesc1, 1u);                              // gy_lo * x_hi
            }
            umma_commit(&empty[s]);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(&acc_full[buf]);
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: TMEM -> fp32 registers -> atomics per item
    constexpr int kCh = BN / 32, kHalf = (kCh + 1) / 2;
    const int lg = warp & 3, half = (warp - 2) >> 2;
    const int row = lg * 32 + lane;                 // TMEM lane = output channel within the co tile
    int t = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
      const Item it = decode(p, item);
      float acc[kHalf * 32];
#pragma unroll
      for (int j = 0; j < kHalf * 32; ++j) acc[j] = 0.f;
      for (long long c0 = it.kb0; c0 < it.kb1; c0 += p.kc, ++t) {
        const int buf = t & 1, use = t >> 1;
        mbar_wait(&acc_full[buf], use & 1);
        tcgen05_fence_after();
#pragma unroll
        for (int i = 0; i < kHalf; ++i) {
          const int c = half * kHalf + i;
          if (c < kCh) {                               // warp-uniform
            uint32_t r[32], rc[32];
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(lg * 32) << 16) + buf * 2 * BN + c * 32;
            tmem_ld32(taddr, r);
            tmem_ld32(taddr + BN, rc);
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[i * 32 + j] += __uint_as_float(r[j]) + __uint_as_float(rc[j]);
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[buf]);
      }
      const int co = it.cot * kBM + row;
      if (co < p.cout) {
        float* dst = p.gw + static_cast<size_t>(it.tap) * p.cin * p.ldw + co;
#pragma unroll
        for (int i = 0; i < kHalf; ++i) {
          const int c = half * kHalf + i;
          if (c >= kCh) break;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int ci = it.cit * BN + c * 32 + j;
            if (ci < p.cin) atomicAdd(dst + static_cast<size_t>(ci) * p.ldw, acc[i * 32 + j]);   // lanes: consecutive co
          }
        }
      }
    }
  }

  // ------------------------------------------------------------------ teardown
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// fp32 CL [B][H][W][ld], channels [0,C) -> TF32 hi/lo planes [B][C][H][Q][pitch]: plane position (q, j) holds input column
// j*S + q - off (zero outside the image), j < Wh.  A block owns 32 channels and walks tiles of 32 plane positions of one
// (image, row, q): reads are 128-byte channel rows, writes 128-byte pixel rows.  gsum (optional; Q = S = 1, off = 0): += sum over
// pixels.
__global__ void __launch_bounds__(256)
plane_split_kernel(const float* __restrict__ src, int ld, int C, int B, int H, int W, int S, int Q, int off, int Wh, int pitch,
                   float* __restrict__ hi, float* __restrict__ lo, float* __restrict__ gsum) {
  __shared__ float tile[32][33];
  __shared__ double red[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c0 = blockIdx.y * 32;
  const int njt = (Wh + 31) / 32;
  const long long ntiles = static_cast<long long>(B) * H * Q * njt;
  double bsum = 0.0;
  for (long long tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
    const int jt = static_cast<int>(tl % njt);
    long long r = tl / njt;
    const int q = static_cast<int>(r % Q);
    r /= Q;
    const int y = static_cast<int>(r % H), b = static_cast<int>(r / H);
    const int j0 = jt * 32;
    float part = 0.f;
#pragma unroll
    for (int i = ty; i < 32; i += 8) {
      const int j = j0 + i, xi = j * S + q - off, c = c0 + tx;
      float v = 0.f;
      if (j < Wh && xi >= 0 && xi < W && c < C) v = __ldg(src + ((static_cast<size_t>(b) * H + y) * W + xi) * ld + c);
      tile[i][tx] = v;
      part += v;
    }
    bsum += static_cast<double>(part);
    __syncthreads();
#pragma unroll
    for (int i = ty; i < 32; i += 8) {
      const int c = c0 + i, j = j0 + tx;
      if (c < C && j < Wh) {
        const float v = tile[tx][i];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
        const size_t o = (((static_cast<size_t>(b) * C + c) * H + y) * Q + q) * pitch + j;
        hi[o] = __uint_as_float(h);
        lo[o] = v - __uint_as_float(h);
      }
    }
    __syncthreads();
  }
  if (gsum != nullptr) {
    red[ty][tx] = bsum;
    __syncthreads();
    if (ty == 0 && c0 + tx < C) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += red[k][tx];
      atomicAdd(gsum + c0 + tx, static_cast<float>(s));
    }
  }
}

// ---------------------------------------------------------------------------------------------- host side
struct Layout {
  int Ho, Wo, pitch;                 // plane rows hold Wo positions, pitch = Wo rounded up to 4 floats (TMA: 16-byte strides)
  size_t xbytes, gbytes;             // one plane each (hi or lo), rounded up to 256 bytes
};

static bool layout(int cin, int cout, int B, int Hin, int Win, int kw, int stride, Layout& L) {
  L.Ho = (Hin + stride - 1) / stride;
  L.Wo = (Win + stride - 1) / stride;
  L.pitch = (L.Wo + 3) / 4 * 4;
  const double xb = 4.0 * B * cin * Hin * kw * L.pitch, gb = 4.0 * B * cout * L.Ho * L.pitch;   // x: one copy per kx
  if (xb > 1e12 || gb > 1e12) return false;
  L.xbytes = (static_cast<size_t>(xb) + 255) / 256 * 256;
  L.gbytes = (static_cast<size_t>(gb) + 255) / 256 * 256;
  return true;
}

// TF32 planes [B][C][H][Q][pitch] floats: 5-D map {Wo, Q, H, C, B}, box = 32 positions x 1 copy x 1 row x rows channels x 1 image
static bool make_plane_map(CUtensorMap* m, const float* base, int Wd, int Q, int H, int C, int B, int pitch, int rows) {
  const cuuint64_t dims[5] = {(cuuint64_t)Wd, (cuuint64_t)Q, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)B};
  const cuuint64_t row = (cuuint64_t)pitch * 4;
  const cuuint64_t strides[4] = {row, row * Q, row * Q * H, row * Q * H * C};
  const cuuint32_t box[5] = {(cuuint32_t)kPx, 1, 1, (cuuint32_t)rows, 1};
  const cuuint32_t es[5] = {1, 1, 1, 1, 1};
  return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

template <int BN>
static int launch(const CUtensorMap* maps, Params& p, cudaStream_t stream) {
  constexpr int kStage = 2 * kAPlane + 2 * BN * 128;
  const int budget = 227 * 1024 - 1024 - 256;      // alignment slack, barriers
  p.stages = budget / kStage < kMaxStages ? budget / kStage : kMaxStages;
  const int smem = p.stages * kStage + 1024 + 256;
  static unsigned long long done = 0;
  if (int st = ensure_dyn_smem(wgrad_umma_kernel<BN>, smem, &done)) return st;
  const int grid = p.items < sm_count() ? p.items : sm_count();
  wgrad_umma_kernel<BN><<<grid, kThreads, smem, stream>>>(maps[0], maps[1], maps[2], maps[3], p);
  return after_launch();
}

}  // namespace wgrad
}  // namespace rnc

using namespace rnc;

extern "C" size_t rnc_conv2d_umma_wgrad_workspace_bytes(int cin, int cout, int B, int Hin, int Win, int kh, int kw, int stride) {
  if (B <= 0 || Hin <= 0 || Win <= 0 || cin <= 0 || cout <= 0 || kh < 1 || kw < 1 || (stride != 1 && stride != 2)) return 0;
  wgrad::Layout L;
  if (!wgrad::layout(cin, cout, B, Hin, Win, kw, stride, L)) return 0;
  return 2 * L.xbytes + 2 * L.gbytes;
}

extern "C" int rnc_conv2d_umma_wgrad(const float* x, int ldx, int cin, const float* gy, int ldg, int cout, int B, int Hin, int Win,
                                     int kh, int kw, int stride, float* gw, int ldw, float* gb, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  using namespace rnc::wgrad;
  if (B <= 0 || Hin <= 0 || Win <= 0 || cin <= 0 || cout <= 0 || (cin & 3) || (ldx & 3) || ldx < cin || ldg < cout || ldw < cout)
    return RNC_ERR_BAD_SHAPE;
  if (kh < 1 || kw < 1 || !(kh & 1) || !(kw & 1) || kh * kw > 49 || (stride != 1 && stride != 2)) return RNC_ERR_BAD_SHAPE;
  if (!x || !gy || !gw || !workspace || !aligned16(x) || !aligned16(gy) || (ldg & 3) || !aligned16(workspace)) return RNC_ERR_BAD_POINTER;
  Layout L;
  if (!layout(cin, cout, B, Hin, Win, kw, stride, L)) return RNC_ERR_UNSUPPORTED;
  if (workspace_bytes < 2 * L.xbytes + 2 * L.gbytes) return RNC_ERR_WORKSPACE;
  if (!umma::encode_fn()) return RNC_ERR_UNSUPPORTED;

  const int nci = (cin + kBM - 1) / kBM;            // ci tiles of at most 128 channels, as even as 32-channel granularity allows
  const int per_tile = (cin + nci - 1) / nci;
  const int bn = (per_tile + 31) / 32 * 32;
  Params p;
  p.Ho = L.Ho; p.nxt = (L.Wo + kPx - 1) / kPx;
  p.kw = kw; p.ph = kh / 2; p.pw = kw / 2; p.stride = stride;
  p.cin = cin; p.cout = cout; p.ldw = ldw;
  p.nco = (cout + kBM - 1) / kBM; p.nci = (cin + bn - 1) / bn; p.taps = kh * kw;
  p.nkb = static_cast<long long>(B) * L.Ho * p.nxt;
  p.gw = gw;
  {
    const char* e = getenv("RNC_WGRAD_KC");       // K blocks (32 px) per chunk: the precision probe of tools/wgrad_probe.py
    p.kc = e != nullptr && atoi(e) > 0 ? atoi(e) : kKC;
  }
  // K splits: fill the SMs, then round the item count up towards whole waves (a finer split of a long K costs only atomics)
  const long long tiles = static_cast<long long>(p.nco) * p.nci * p.taps, sms = sm_count();
  const long long max_ks = (p.nkb + kMinPer - 1) / kMinPer;
  long long nks = (sms + tiles - 1) / tiles;
  if (nks > max_ks) nks = max_ks;
  if (nks < 1) nks = 1;
  const long long rounds = (tiles * nks + sms - 1) / sms;
  if (rounds * sms / tiles > nks) nks = rounds * sms / tiles < max_ks ? rounds * sms / tiles : max_ks;
  p.per = (p.nkb + nks - 1) / nks;
  nks = (p.nkb + p.per - 1) / p.per;
  if (tiles * nks > (1LL << 30)) return RNC_ERR_UNSUPPORTED;
  p.items = static_cast<int>(tiles * nks);

  unsigned char* ws = static_cast<unsigned char*>(workspace);
  float* xh = reinterpret_cast<float*>(ws);
  float* xl = reinterpret_cast<float*>(ws + L.xbytes);
  float* gh = reinterpret_cast<float*>(ws + 2 * L.xbytes);
  float* gl = reinterpret_cast<float*>(ws + 2 * L.xbytes + L.gbytes);
  CUtensorMap maps[4];
  if (!make_plane_map(&maps[0], gh, L.Wo, 1, L.Ho, cout, B, L.pitch, kBM) || !make_plane_map(&maps[1], gl, L.Wo, 1, L.Ho, cout, B, L.pitch, kBM) ||
      !make_plane_map(&maps[2], xh, L.Wo, kw, Hin, cin, B, L.pitch, bn) || !make_plane_map(&maps[3], xl, L.Wo, kw, Hin, cin, B, L.pitch, bn))
    return RNC_ERR_UNSUPPORTED;

  cudaStream_t s = as_stream(stream);
  auto split = [&](const float* src, int ld, int C, int H, int W, int S, int Q, int off, float* hi, float* lo, float* sum) {
    const int cy = (C + 31) / 32;
    const long long nt = static_cast<long long>(B) * H * Q * ((L.Wo + 31) / 32);
    long long gx = (sms * 16 + cy - 1) / cy;
    if (gx > nt) gx = nt;
    plane_split_kernel<<<dim3(static_cast<unsigned>(gx), cy), 256, 0, s>>>(src, ld, C, B, H, W, S, Q, off, L.Wo, L.pitch, hi, lo, sum);
    return after_launch();
  };
  if (int st = split(gy, ldg, cout, L.Ho, L.Wo, 1, 1, 0, gh, gl, gb)) return st;
  if (int st = split(x, ldx, cin, Hin, Win, stride, kw, kw / 2, xh, xl, nullptr)) return st;
  switch (bn) {
    case 32: return launch<32>(maps, p, s);
    case 64: return launch<64>(maps, p, s);
    case 96: return launch<96>(maps, p, s);
    default: return launch<128>(maps, p, s);
  }
}
