// Layout plumbing: NCHW <-> channel-last, feature pyramid, coordinate grid.
// Replaces: core/corr.py:7-21 (pyramid construction, here on features instead of on the 4-D volume),
//           core/utils/utils.py:76-79 (coords_grid), raft_nc_dbl.py:83-90,144-145,152.
#include "rnc_common.cuh"

namespace rnc {

thread_local int g_last_cuda_error = 0;
thread_local long long g_launch_count = 0;

// src [B][C][P]  ->  dst [B][P][ld] (+ch_off)
__global__ void nchw_to_cl_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int P, int ld, int ch_off) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* s = src + (size_t)b * C * P;
  float* d = dst + (size_t)b * P * ld + ch_off;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int c = c0 + i, p = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && p < P) ? s[(size_t)c * P + p] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    int p = p0 + i, c = c0 + threadIdx.x;
    if (p < P && c < C) d[(size_t)p * ld + c] = tile[threadIdx.x][i];
  }
}

// src [B][P][ld] (+ch_off)  ->  dst [B][C][P]
__global__ void cl_to_nchw_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int P, int ld, int ch_off) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* s = src + (size_t)b * P * ld + ch_off;
  float* d = dst + (size_t)b * C * P;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int p = p0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && p < P) ? s[(size_t)p * ld + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    int c = c0 + i, p = p0 + threadIdx.x;
    if (p < P && c < C) d[(size_t)c * P + p] = tile[threadIdx.x][i];
  }
}

// 2x2 floor-mode average pool on a CL tensor: src [B][Hs][Ws][D] -> dst [B][Hs/2][Ws/2][D]; one float4 per thread.
__global__ void pool2_cl_kernel(const float4* __restrict__ src, float4* __restrict__ dst, int B, int Hs, int Ws, int D4) {
  const int Hd = Hs >> 1, Wd = Ws >> 1;
  size_t n = (size_t)B * Hd * Wd * D4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    int d = (int)(i % D4);
    size_t r = i / D4;
    int x = (int)(r % Wd); r /= Wd;
    int y = (int)(r % Hd);
    int b = (int)(r / Hd);
    const float4* s = src + (((size_t)b * Hs + 2 * y) * Ws + 2 * x) * D4 + d;
    float4 a = s[0], c = s[D4], e = s[(size_t)Ws * D4], f = s[(size_t)Ws * D4 + D4];
    float4 o;
    o.x = 0.25f * ((a.x + c.x) + (e.x + f.x));
    o.y = 0.25f * ((a.y + c.y) + (e.y + f.y));
    o.z = 0.25f * ((a.z + c.z) + (e.z + f.z));
    o.w = 0.25f * ((a.w + c.w) + (e.w + f.w));
    dst[i] = o;
  }
}

__global__ void coords_init_kernel(float* __restrict__ coords1, const float* __restrict__ flow_init, int B, int H, int W) {
  int n = B * 2 * H * W;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int x = i % W, y = (i / W) % H, c = (i / (W * H)) % 2;
    float g = c == 0 ? (float)x : (float)y;
    coords1[i] = flow_init ? g + flow_init[i] : g;
  }
}

__global__ void coords_to_flow_kernel(const float* __restrict__ coords1, float* __restrict__ flow, int B, int H, int W) {
  int n = B * 2 * H * W;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int x = i % W, y = (i / W) % H, c = (i / (W * H)) % 2;
    flow[i] = coords1[i] - (c == 0 ? (float)x : (float)y);
  }
}

}  // namespace rnc

using namespace rnc;

extern "C" {

int rnc_abi_version(void) { return 11; }
const char* rnc_build_info(void) { return "librnc sm_100a (CUDA " RNC_STR_CUDA ")"; }
const char* rnc_status_string(int s) {
  switch (s) {
    case RNC_OK: return "ok";
    case RNC_ERR_BAD_SHAPE: return "bad shape";
    case RNC_ERR_BAD_POINTER: return "null or misaligned pointer";
    case RNC_ERR_UNSUPPORTED: return "unsupported configuration";
    case RNC_ERR_CUDA: return "CUDA launch error";
    case RNC_ERR_WORKSPACE: return "workspace too small";
  }
  return "unknown status";
}
int rnc_last_cuda_error(void) { return g_last_cuda_error; }
long long rnc_launch_count(void) { return g_launch_count; }
void rnc_launch_count_reset(void) { g_launch_count = 0; }

size_t rnc_pyramid_offset(int B, int D, int H, int W, int level) {
  size_t off = 0;
  for (int l = 0; l < level; ++l) off += (size_t)B * (H >> l) * (W >> l) * D;
  return off;
}

int rnc_nchw_to_cl(const float* src, int B, int C, int H, int W, float* dst, int ldd, int ch_off, void* stream) {
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || ldd < C + ch_off || ch_off < 0) return RNC_ERR_BAD_SHAPE;
  if (!src || !dst) return RNC_ERR_BAD_POINTER;
  int P = H * W;
  dim3 grid((P + 31) / 32, (C + 31) / 32, B), block(32, 8);
  nchw_to_cl_kernel<<<grid, block, 0, as_stream(stream)>>>(src, dst, C, P, ldd, ch_off);
  return after_launch();
}

int rnc_cl_to_nchw(const float* src, int lds, int ch_off, int B, int C, int H, int W, float* dst, void* stream) {
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || lds < C + ch_off || ch_off < 0) return RNC_ERR_BAD_SHAPE;
  if (!src || !dst) return RNC_ERR_BAD_POINTER;
  int P = H * W;
  dim3 grid((P + 31) / 32, (C + 31) / 32, B), block(32, 8);
  cl_to_nchw_kernel<<<grid, block, 0, as_stream(stream)>>>(src, dst, C, P, lds, ch_off);
  return after_launch();
}

int rnc_fmap_prepare(const float* fmap1, const float* fmap2, int B, int D, int H, int W, int levels,
                     float* f1_cl, float* f2_pyr, void* stream) {
  if (B <= 0 || D <= 0 || (D & 3) || H <= 0 || W <= 0 || levels < 1 || levels > 4) return RNC_ERR_BAD_SHAPE;
  if ((H >> (levels - 1)) < 1 || (W >> (levels - 1)) < 1) return RNC_ERR_BAD_SHAPE;
  if (!fmap1 || !fmap2 || !f1_cl || !f2_pyr || !aligned16(f1_cl) || !aligned16(f2_pyr)) return RNC_ERR_BAD_POINTER;
  int st = rnc_nchw_to_cl(fmap1, B, D, H, W, f1_cl, D, 0, stream);
  if (st) return st;
  st = rnc_nchw_to_cl(fmap2, B, D, H, W, f2_pyr, D, 0, stream);
  if (st) return st;
  for (int l = 1; l < levels; ++l) {
    const float* s = f2_pyr + rnc_pyramid_offset(B, D, H, W, l - 1);
    float* d = f2_pyr + rnc_pyramid_offset(B, D, H, W, l);
    int Hs = H >> (l - 1), Ws = W >> (l - 1);
    size_t n = (size_t)B * (Hs >> 1) * (Ws >> 1) * (D / 4);
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    pool2_cl_kernel<<<blocks, 256, 0, as_stream(stream)>>>((const float4*)s, (float4*)d, B, Hs, Ws, D / 4);
    st = after_launch();
    if (st) return st;
  }
  return RNC_OK;
}

int rnc_coords_init(float* coords1, const float* flow_init, int B, int H, int W, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0) return RNC_ERR_BAD_SHAPE;
  if (!coords1) return RNC_ERR_BAD_POINTER;
  int n = B * 2 * H * W;
  coords_init_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(coords1, flow_init, B, H, W);
  return after_launch();
}

int rnc_coords_to_flow(const float* coords1, float* flow, int B, int H, int W, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0) return RNC_ERR_BAD_SHAPE;
  if (!coords1 || !flow) return RNC_ERR_BAD_POINTER;
  int n = B * 2 * H * W;
  coords_to_flow_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(coords1, flow, B, H, W);
  return after_launch();
}

}  // extern "C"
