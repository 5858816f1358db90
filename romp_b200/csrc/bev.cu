// BEV-specific stages of the hot path (BASELINE.json configs[2]): everything of simple_romp/bev/model.py and
// bev/post_parser.py that is not a 2-D / 1-D convolution (those run on the conv-graph engines).
//
//   bev_bv_input      : torch.cat([center_fv, cam_offset, img_feats],1).view(B,-1,128)           bev/model.py:190
//   bev_center3d      : outer product fv x bv + BasicBlock_3D(1->1) refiner                       :195-196,206 (+:52-75)
//   bev_parse3d       : CenterMap3D.parse_3dcentermap (5x5x5 max-pool NMS, top-64, threshold)     bev/post_parser.py:44-66
//   bev_regress       : cam_maps_3d sampled at the detections - evaluated LAZILY: the BasicBlock_3D(3->3) refiner is
//                       computed only on the 5^3 neighbourhood of each detection instead of materialising the
//                       [B,3,64,128,128] volume (12.6 MB/frame) - then anchor arg-min, feature sampling + position
//                       embedding and the 128-512-512-143 MLP                                     bev/model.py:209-213,217-230,242
//   bev_unpack        : pack_params_dict (11 betas) + denormalize_cam_params_to_trans             bev/post_parser.py:240-253,114-128
//   bev_merge_smil    : SMPLA_parser's baby/adult split (betas[:,10] > 0.8)                       :255-278
//   bev_project       : perspective_projection (f=443.4) + convert to original-image pixels       :68-107,129-152
//   bev_postfilter    : suppressing_redundant_prediction_via_projection + remove_outlier, applied per frame
//                       (the reference assumes one frame)                                         :167-222
// All fp32, one host sync per batch (the final person count).
#include <math_constants.h>

#include <vector>

#include "common.cuh"
#include "rot6d.cuh"

namespace b200romp {

constexpr int kD = 64, kS = 128, kVol = kD * kS * kS;
constexpr int kCandCap = 4096;          // local maxima above threshold kept per frame before the top-64 sort
constexpr int kMaxP = 64;
constexpr float kTanFov = 0.57735026919f;   // tan(radians(60/2)), bev/post_parser.py:109

struct BevDev {
  const float* center_ref;   // [56]  w1[27] b1 w2[27] b2   (BatchNorm3d folded)
  const float* cam_ref;      // [492] w1[3][3][27] b1[3] w2[3][3][27] b2[3]
  const float* coordmap;     // [64][128][128][3]
  const float* anchors;      // [64]
  const float* embed;        // [128][128]
  const float *w0t, *b0, *w1t, *b1, *w2t, *b2;   // MLP, weights transposed to [in][out]
};

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bev_bv_input_kernel(const float* __restrict__ maps_fv, const void* __restrict__ feats,
                                                           int feats_dtype, int feats_C, int B, void* __restrict__ out, int out_dtype) {
  const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (size_t)B * kS * 2560) return;
  const int ch = idx % 2560, w = (idx / 2560) % kS, b = idx / ((size_t)2560 * kS);
  const int c = ch / kS, h = ch % kS;
  float v;
  if (c < 4) v = maps_fv[(((size_t)b * 4 + c) * kS + h) * kS + w];
  else v = load_as_float(feats, (((size_t)b * kS + h) * kS + w) * feats_C + (c - 4), feats_dtype);
  store_from_float(out, idx, out_dtype, v);
}

// center_map_3d = fv (x) bv, refined by BasicBlock_3D(1->1).  stage 1: t1 = relu(bn1(conv1(cm))); stage 2: bn2(conv2(t1)) + cm
__device__ __forceinline__ float cm_at(const float* cfv, const void* bv, int bv_dtype, int b, int d, int h, int w) {
  return cfv[((size_t)b * 4 * kS + h) * kS + w] * load_as_float(bv, ((size_t)b * kS + w) * kS + d, bv_dtype);
}

__global__ void __launch_bounds__(256) bev_center3d_kernel(const float* __restrict__ maps_fv, const void* __restrict__ bv,
                                                           int bv_dtype, BevDev m, int B, const float* __restrict__ t1,
                                                           float* __restrict__ out, int stage) {
  const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (size_t)B * kVol) return;
  const int w = idx % kS, h = (idx / kS) % kS, d = (idx / (kS * kS)) % kD, b = idx / kVol;
  const float* wgt = m.center_ref + (stage == 1 ? 0 : 28);
  float acc = wgt[27];
#pragma unroll
  for (int dz = -1; dz <= 1; ++dz)
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
      for (int dx = -1; dx <= 1; ++dx) {
        const int zz = d + dz, yy = h + dy, xx = w + dx;
        if (zz < 0 || zz >= kD || yy < 0 || yy >= kS || xx < 0 || xx >= kS) continue;
        const float x = stage == 1 ? cm_at(maps_fv, bv, bv_dtype, b, zz, yy, xx)
                                   : t1[(((size_t)b * kD + zz) * kS + yy) * kS + xx];
        acc = fmaf(wgt[(dz + 1) * 9 + (dy + 1) * 3 + (dx + 1)], x, acc);
      }
  out[idx] = stage == 1 ? fmaxf(acc, 0.f) : acc + cm_at(maps_fv, bv, bv_dtype, b, d, h, w);
}

// Fused version of the two stages above (round 2): one kernel, the intermediate t1 never leaves shared memory, and stage 1
// uses the rank-1 structure of its input: cm[d,h,w] = fv[h,w] * bv[w,d], so
//     conv1(cm)[d,h,w] = sum_{a,c} bv[w+c, d+a] * G[a,c][h, w+c],   G[a,c][h,x] = sum_b k1[a,b,c] * fv[h+b, x]
// (9 FMA per voxel instead of 27; G is 9 planes of the block's 10 x 36 footprint).  Stage 2 is the full 27-tap stencil on the
// shared-memory t1 tile with a sliding window along d.  Block = 8 (d) x 8 (h) x 32 (w) outputs, 256 threads.
// FLOPs per output: 9 * (10*10*34)/(8*8*32) + 27 = 42 (was 54), global traffic: one fp32 store per voxel (was 3 accesses).
constexpr int kTD = 8, kTH = 8, kTW = 32;
__global__ void __launch_bounds__(256) bev_center3d_fused_kernel(const float* __restrict__ maps_fv, const void* __restrict__ bv,
                                                                 int bv_dtype, BevDev m, float* __restrict__ out) {
  __shared__ float s_fv[kTH + 4][kTW + 4];            // fv rows h0-2 .. h0+9, cols w0-2 .. w0+33 (zero outside the map)
  __shared__ float s_bv[kTW + 4][kTD + 4];            // bv[w][d] cols w0-2.., depth d0-2 .. d0+9 (zero outside)
  __shared__ float s_G[9][kTH + 2][kTW + 4];          // G[a*3+c][h0-1 .. h0+8][w0-2 .. w0+33]
  __shared__ float s_t1[kTD + 2][kTH + 2][kTW + 2];   // relu(conv1 + b1) on the halo tile, zero outside the volume
  const int b = blockIdx.z;
  const int w0 = (blockIdx.x % (kS / kTW)) * kTW, h0 = (blockIdx.x / (kS / kTW)) * kTH, d0 = blockIdx.y * kTD;
  const int tid = threadIdx.x;
  const float* cfv = maps_fv + (size_t)b * 4 * kS * kS;            // channel 0 = center_maps_fv
  for (int i = tid; i < (kTH + 4) * (kTW + 4); i += 256) {
    const int r = i / (kTW + 4), c = i % (kTW + 4), h = h0 - 2 + r, w = w0 - 2 + c;
    s_fv[r][c] = (h >= 0 && h < kS && w >= 0 && w < kS) ? cfv[(size_t)h * kS + w] : 0.f;
  }
  for (int i = tid; i < (kTW + 4) * (kTD + 4); i += 256) {
    const int c = i / (kTD + 4), r = i % (kTD + 4), w = w0 - 2 + c, d = d0 - 2 + r;
    s_bv[c][r] = (w >= 0 && w < kS && d >= 0 && d < kD) ? load_as_float(bv, ((size_t)b * kS + w) * kS + d, bv_dtype) : 0.f;
  }
  __syncthreads();
  const float* k1 = m.center_ref;                       // [27] then b1
  for (int i = tid; i < 9 * (kTH + 2) * (kTW + 4); i += 256) {
    const int x = i % (kTW + 4), r = (i / (kTW + 4)) % (kTH + 2), ac = i / ((kTW + 4) * (kTH + 2));
    const int a = ac / 3, c = ac % 3;
    // G[a,c][h0-1+r][w0-2+x] = sum_b k1[a][b][c] * fv[h0-1+r + (b-1)][.]  (s_fv row index = r + b)
    s_G[ac][r][x] = k1[a * 9 + 0 * 3 + c] * s_fv[r + 0][x] + k1[a * 9 + 1 * 3 + c] * s_fv[r + 1][x] + k1[a * 9 + 2 * 3 + c] * s_fv[r + 2][x];
  }
  __syncthreads();
  const float b1 = k1[27];
  for (int i = tid; i < (kTH + 2) * (kTW + 2); i += 256) {      // one (h, w) column of the t1 halo tile per iteration
    const int wl = i % (kTW + 2), hl = i / (kTW + 2);            // t1 position (h0-1+hl, w0-1+wl); s_G / s_bv column index = wl + 1 + (c-1)
    const int h = h0 - 1 + hl, w = w0 - 1 + wl;
    const bool inside_hw = h >= 0 && h < kS && w >= 0 && w < kS;
    float g[9];
#pragma unroll
    for (int ac = 0; ac < 9; ++ac) g[ac] = s_G[ac][hl][wl + (ac % 3)];
#pragma unroll
    for (int dl = 0; dl < kTD + 2; ++dl) {                       // t1 depth d0-1+dl; s_bv depth index = dl + 1 + (a-1)
      float acc = b1;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) acc = fmaf(s_bv[wl + c][dl + a], g[a * 3 + c], acc);
      const int d = d0 - 1 + dl;
      s_t1[dl][hl][wl] = (inside_hw && d >= 0 && d < kD) ? fmaxf(acc, 0.f) : 0.f;
    }
  }
  __syncthreads();
  const float* k2 = m.center_ref + 28;                  // [27] then b2
  float wk[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) wk[i] = k2[i];
  const float b2 = k2[27];
  const int wl = tid % kTW, hl = tid / kTW;             // output (h0+hl, w0+wl), all kTD depths
  float p0[9], p1[9], p2[9];                            // t1 planes d-1, d, d+1 (3x3 in h, w)
#pragma unroll
  for (int j = 0; j < 9; ++j) { p0[j] = s_t1[0][hl + j / 3][wl + j % 3]; p1[j] = s_t1[1][hl + j / 3][wl + j % 3]; }
  const float fvv = s_fv[hl + 2][wl + 2];
#pragma unroll
  for (int dl = 0; dl < kTD; ++dl) {
#pragma unroll
    for (int j = 0; j < 9; ++j) p2[j] = s_t1[dl + 2][hl + j / 3][wl + j % 3];
    float acc = b2;
#pragma unroll
    for (int j = 0; j < 9; ++j) acc = fmaf(wk[j], p0[j], acc);
#pragma unroll
    for (int j = 0; j < 9; ++j) acc = fmaf(wk[9 + j], p1[j], acc);
#pragma unroll
    for (int j = 0; j < 9; ++j) acc = fmaf(wk[18 + j], p2[j], acc);
    const float cm = fvv * s_bv[wl + 2][dl + 2];
    out[(((size_t)b * kD + d0 + dl) * kS + h0 + hl) * kS + w0 + wl] = acc + cm;
#pragma unroll
    for (int j = 0; j < 9; ++j) { p0[j] = p1[j]; p1[j] = p2[j]; }
  }
}

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bev_nms3d_kernel(const float* __restrict__ c3d, int B, float thresh,
                                                        int* __restrict__ cand_count, int* __restrict__ cand_idx,
                                                        float* __restrict__ cand_val) {
  const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (size_t)B * kVol) return;
  const float v = c3d[idx];
  if (!(v > thresh)) return;                       // det * (maxpool == det) > thresh  <=>  det > thresh and det is a maximum
  const int vox = idx % kVol, b = idx / kVol;
  const int x = vox % kS, y = (vox / kS) % kS, z = vox / (kS * kS);
  const float* base = c3d + (size_t)b * kVol;
  for (int dz = -2; dz <= 2; ++dz) {
    const int zz = z + dz;
    if (zz < 0 || zz >= kD) continue;
    for (int dy = -2; dy <= 2; ++dy) {
      const int yy = y + dy;
      if (yy < 0 || yy >= kS) continue;
      for (int dx = -2; dx <= 2; ++dx) {
        const int xx = x + dx;
        if (xx < 0 || xx >= kS) continue;
        if (base[((size_t)zz * kS + yy) * kS + xx] > v) return;
      }
    }
  }
  const int slot = atomicAdd(&cand_count[b], 1);
  if (slot < kCandCap) {
    cand_idx[(size_t)b * kCandCap + slot] = vox;
    cand_val[(size_t)b * kCandCap + slot] = v;
  }
}

__device__ __forceinline__ bool before3(float ka, int ia, float kb, int ib) { return (ka > kb) || (ka == kb && ia < ib); }

__global__ void __launch_bounds__(1024) bev_top64_kernel(const int* __restrict__ cand_count, const int* __restrict__ cand_idx,
                                                         const float* __restrict__ cand_val, int* __restrict__ counts,
                                                         int* __restrict__ top_idx, float* __restrict__ top_val) {
  __shared__ float s_key[kCandCap];
  __shared__ int s_idx[kCandCap];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = min(cand_count[b], kCandCap);
  for (int i = tid; i < kCandCap; i += 1024) {
    s_key[i] = i < n ? cand_val[(size_t)b * kCandCap + i] : -CUDART_INF_F;
    s_idx[i] = i < n ? cand_idx[(size_t)b * kCandCap + i] : 0x7fffffff;
  }
  __syncthreads();
  for (int k = 2; k <= kCandCap; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < kCandCap / 2; t += 1024) {
        const int lo = ((t / j) * 2 * j) + (t % j), hi = lo + j;
        const bool up = ((lo & k) == 0);
        const float ka = s_key[lo], kb = s_key[hi];
        const int ia = s_idx[lo], ib = s_idx[hi];
        if (before3(ka, ia, kb, ib) != up) {
          s_key[lo] = kb; s_key[hi] = ka; s_idx[lo] = ib; s_idx[hi] = ia;
        }
      }
      __syncthreads();
    }
  if (tid < kMaxP) {
    top_idx[b * kMaxP + tid] = s_idx[tid];
    top_val[b * kMaxP + tid] = s_key[tid];
  }
  if (tid == 0) counts[b] = min(n, kMaxP);
}

__global__ void __launch_bounds__(64) bev_emit_kernel(int B, int capacity, const int* __restrict__ counts,
                                                      const int* __restrict__ top_idx, const float* __restrict__ top_val,
                                                      int* __restrict__ d_count, long long* __restrict__ batch_ids,
                                                      long long* __restrict__ czyx, float* __restrict__ conf) {
  const int b = blockIdx.x, tid = threadIdx.x;
  __shared__ int s_off;
  if (tid == 0) {
    int o = 0;
    for (int i = 0; i < b; ++i) o += counts[i];
    s_off = o;
    if (b == B - 1) *d_count = min(o + counts[b], capacity);
  }
  __syncthreads();
  const int n = s_off + tid;
  if (tid < counts[b] && n < capacity) {
    const int vox = top_idx[b * kMaxP + tid];
    batch_ids[n] = b;
    czyx[(size_t)n * 3 + 0] = vox / (kS * kS);
    czyx[(size_t)n * 3 + 1] = (vox / kS) % kS;
    czyx[(size_t)n * 3 + 2] = vox % kS;
    conf[n] = top_val[b * kMaxP + tid];
  }
}

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bev_regress_kernel(BevDev m, const float* __restrict__ maps_fv, const void* __restrict__ bv,
                                                          int bv_dtype, const void* __restrict__ fv, int fv_dtype,
                                                          const int* __restrict__ d_count, const long long* __restrict__ batch_ids,
                                                          const long long* __restrict__ czyx, float* __restrict__ params_pred,
                                                          long long* __restrict__ cam_czyx) {
  const int n = blockIdx.x, tid = threadIdx.x;
  if (n >= *d_count) return;
  __shared__ float s_in[3][125];
  __shared__ float s_t1[3][27];
  __shared__ float s_cam[3];
  __shared__ int s_c[3];
  __shared__ float s_f[128], s_h1[512], s_h2[512];
  const int b = (int)batch_ids[n], z = (int)czyx[n * 3], y = (int)czyx[n * 3 + 1], x = (int)czyx[n * 3 + 2];
  // cam_maps_3d input field on the 5^3 neighbourhood: coordmap + cam_offset (+ bird's-eye offset on the last component)
  for (int t = tid; t < 375; t += 256) {
    const int c = t / 125, r = t % 125;
    const int zz = z + r / 25 - 2, yy = y + (r / 5) % 5 - 2, xx = x + r % 5 - 2;
    float v = 0.f;                                                  // zero padding of the 3-D conv
    if (zz >= 0 && zz < kD && yy >= 0 && yy < kS && xx >= 0 && xx < kS) {
      v = m.coordmap[(((size_t)zz * kS + yy) * kS + xx) * 3 + c] + maps_fv[(((size_t)b * 4 + 1 + c) * kS + yy) * kS + xx];
      if (c == 2) v += load_as_float(bv, ((size_t)b * kS + xx) * kS + 64 + zz, bv_dtype);   // bev/model.py:212
    }
    s_in[c][r] = v;
  }
  __syncthreads();
  if (tid < 81) {       // t1 = relu(bn1(conv1)) at the 27 neighbours (zero outside the volume: conv2's padding)
    const int c1 = tid / 27, nb = tid % 27;
    const int nz = nb / 9 - 1, ny = (nb / 3) % 3 - 1, nx = nb % 3 - 1;
    float acc = 0.f;
    if (z + nz >= 0 && z + nz < kD && y + ny >= 0 && y + ny < kS && x + nx >= 0 && x + nx < kS) {
      acc = m.cam_ref[243 + c1];
      for (int c0 = 0; c0 < 3; ++c0)
        for (int tz = 0; tz < 3; ++tz)
          for (int ty = 0; ty < 3; ++ty)
            for (int tx = 0; tx < 3; ++tx)
              acc = fmaf(m.cam_ref[(c1 * 3 + c0) * 27 + tz * 9 + ty * 3 + tx],
                         s_in[c0][(nz + tz + 1) * 25 + (ny + ty + 1) * 5 + (nx + tx + 1)], acc);
      acc = fmaxf(acc, 0.f);
    }
    s_t1[c1][nb] = acc;
  }
  __syncthreads();
  if (tid < 3) {
    float acc = m.cam_ref[489 + tid];
    for (int c1 = 0; c1 < 3; ++c1)
      for (int t = 0; t < 27; ++t) acc = fmaf(m.cam_ref[246 + (tid * 3 + c1) * 27 + t], s_t1[c1][t], acc);
    s_cam[tid] = acc + s_in[tid][62];                                 // residual of BasicBlock_3D, centre voxel
  }
  __syncthreads();
  if (tid == 0) {       // convert_cam_params_to_centermap_coords + denormalize_center, bev/model.py:89-102
    int best = 0;
    float bd = fabsf(s_cam[0] - m.anchors[0]);
    for (int k = 1; k < 64; ++k) {
      const float dd = fabsf(s_cam[0] - m.anchors[k]);
      if (dd < bd) { bd = dd; best = k; }
    }
    const float c0 = (((float)best / 128.f * 2.f - 1.f) + 1.f) / 2.f * 128.f;
    const float c1 = (s_cam[1] + 1.f) / 2.f * 128.f, c2 = (s_cam[2] + 1.f) / 2.f * 128.f;
    s_c[0] = (int)fminf(fmaxf(c0, 1.f), 127.f);
    s_c[1] = (int)fminf(fmaxf(c1, 1.f), 127.f);
    s_c[2] = (int)fminf(fmaxf(c2, 1.f), 127.f);
    cam_czyx[n * 3] = s_c[0]; cam_czyx[n * 3 + 1] = s_c[1]; cam_czyx[n * 3 + 2] = s_c[2];
  }
  __syncthreads();
  if (tid < 128)       // feature[b,:,cy,cx] + position_embeddings(cz), bev/model.py:217-223
    s_f[tid] = load_as_float(fv, (((size_t)b * kS + s_c[1]) * kS + s_c[2]) * 128 + tid, fv_dtype) + m.embed[s_c[0] * 128 + tid];
  __syncthreads();
  for (int j = tid; j < 512; j += 256) {
    float acc = m.b0[j];
    for (int k = 0; k < 128; ++k) acc = fmaf(m.w0t[k * 512 + j], s_f[k], acc);
    s_h1[j] = fmaxf(acc, 0.f);
  }
  __syncthreads();
  for (int j = tid; j < 512; j += 256) {
    float acc = m.b1[j];
    for (int k = 0; k < 512; ++k) acc = fmaf(m.w1t[k * 512 + j], s_h1[k], acc);
    s_h2[j] = fmaxf(acc, 0.f);
  }
  __syncthreads();
  if (tid < 143) {
    float acc = m.b2[tid];
    for (int k = 0; k < 512; ++k) acc = fmaf(m.w2t[k * 143 + tid], s_h2[k], acc);
    params_pred[(size_t)n * 146 + 3 + tid] = acc;
  }
  if (tid < 3) params_pred[(size_t)n * 146 + tid] = s_cam[tid];
}

__global__ void __launch_bounds__(64) bev_unpack_kernel(const float* __restrict__ params_pred, const int* __restrict__ d_count,
                                                        float* __restrict__ cam, float* __restrict__ thetas,
                                                        float* __restrict__ betas, float* __restrict__ cam_trans) {
  const int n = blockIdx.x, tid = threadIdx.x;
  if (n >= *d_count) return;
  __shared__ float s_row[146];
  for (int i = tid; i < 146; i += 64) s_row[i] = params_pred[(size_t)n * 146 + i];
  __syncthreads();
  if (tid < 22) {
    float aa[3];
    rot6d_to_aa(&s_row[3 + tid * 6], aa);
    thetas[(size_t)n * 72 + tid * 3] = aa[0]; thetas[(size_t)n * 72 + tid * 3 + 1] = aa[1]; thetas[(size_t)n * 72 + tid * 3 + 2] = aa[2];
  } else if (tid < 28) {
    thetas[(size_t)n * 72 + 66 + tid - 22] = 0.f;
  } else if (tid < 31) {
    cam[n * 3 + tid - 28] = s_row[tid - 28];
  } else if (tid >= 32 && tid < 43) {
    betas[(size_t)n * 11 + tid - 32] = s_row[135 + tid - 32];
  } else if (tid == 48) {       // denormalize_cam_params_to_trans, bev/post_parser.py:114-128
    const float depth = 1.f / (s_row[0] * kTanFov + 1e-3f);
    cam_trans[n * 3 + 0] = s_row[2] * depth * kTanFov;
    cam_trans[n * 3 + 1] = s_row[1] * depth * kTanFov;
    cam_trans[n * 3 + 2] = depth;
  }
}

__global__ void __launch_bounds__(256) bev_merge_smil_kernel(const float* __restrict__ betas, const int* __restrict__ d_count,
                                                             const float* __restrict__ verts_smil, const float* __restrict__ joints_smil,
                                                             float* __restrict__ verts, float* __restrict__ joints) {
  const int n = blockIdx.x;
  if (n >= *d_count || !(betas[(size_t)n * 11 + 10] > 0.8f)) return;      // baby_thresh, bev/post_parser.py:260,263
  for (int i = blockIdx.y * 256 + threadIdx.x; i < 6890 * 3; i += gridDim.y * 256) verts[(size_t)n * 20670 + i] = verts_smil[(size_t)n * 20670 + i];
  if (blockIdx.y == 0)
    for (int i = threadIdx.x; i < 213; i += 256) joints[(size_t)n * 213 + i] = joints_smil[(size_t)n * 213 + i];
}

__global__ void __launch_bounds__(128) bev_project_kernel(const float* __restrict__ joints, const float* __restrict__ cam_trans,
                                                          const int* __restrict__ d_count, float size, float left, float top,
                                                          float* __restrict__ pj2d_org) {
  const int n = blockIdx.x, j = threadIdx.x;
  if (n >= *d_count || j >= 71) return;
  const float* q = joints + ((size_t)n * 71 + j) * 3;
  const float px = q[0] + cam_trans[n * 3], py = q[1] + cam_trans[n * 3 + 1], pz = q[2] + cam_trans[n * 3 + 2];
  const float iz = pz + 1e-6f;
  const float u = (px / iz) * 443.4f / 256.f, v = (py / iz) * 443.4f / 256.f;     // bev/post_parser.py:95-105
  pj2d_org[((size_t)n * 71 + j) * 2 + 0] = (u + 1.f) * size / 2.f - left;          // :132-133
  pj2d_org[((size_t)n * 71 + j) * 2 + 1] = (v + 1.f) * size / 2.f - top;
}

// one CTA per frame: both reference post-filters on that frame's (<= 64) persons, then flags for the survivors.
// conf == NULL: the duplicate with the smaller scale goes (bev/post_parser.py:195); else the one with the lower centre
// confidence (conf_based, :191-193, crowd mode).  valid == NULL: every person of the frame takes part; else only those with
// valid[n] != 0 (crowd mode's boundary exclusion ran first), the others keep their 0 flag.
__global__ void __launch_bounds__(256) bev_postfilter_kernel(const float* __restrict__ pj2d_org, const float* __restrict__ cam,
                                                             const float* __restrict__ cam_trans, const long long* __restrict__ batch_ids,
                                                             const int* __restrict__ d_count, float nms_thr_px, float rel_scale_thresh,
                                                             const float* __restrict__ conf, float scale_thresh,
                                                             const int* __restrict__ valid, int* __restrict__ keep) {
  __shared__ int s_n;
  __shared__ int s_idx[kMaxP], s_removed[kMaxP], s_kept[kMaxP], s_nk;
  __shared__ float s_mean[kMaxP];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int N = *d_count;
  if (tid == 0) {
    int s = 0;
    while (s < N && batch_ids[s] < b) ++s;
    int k = 0;
    for (int e = s; e < N && batch_ids[e] == b && k < kMaxP; ++e)
      if (!valid || valid[e]) s_idx[k++] = e;
    s_n = k;
  }
  if (tid < kMaxP) s_removed[tid] = 0;
  __syncthreads();
  const int nf = s_n;
  if (nf == 0) return;
  if (nf > 1) {       // suppressing_redundant_prediction_via_projection, bev/post_parser.py:167-198
    for (int pr = tid; pr < nf * nf; pr += 256) {
      const int i = pr / nf, j = pr % nf;
      if (i >= j) continue;
      const int ni = s_idx[i], nj = s_idx[j];
      const float* a = pj2d_org + (size_t)ni * 142;
      const float* c = pj2d_org + (size_t)nj * 142;
      float sum = 0.f;
      for (int k = 0; k < 71; ++k) {
        const float dx = a[2 * k] - c[2 * k], dy = a[2 * k + 1] - c[2 * k + 1];
        sum += sqrtf(dx * dx + dy * dy);
      }
      const float si = cam[ni * 3] * 2.f, sj = cam[nj * 3] * 2.f;
      const bool lose_i = conf ? conf[ni] < conf[nj] : si < sj;
      if (sum / 71.f / fmaxf(si, sj) < nms_thr_px) atomicExch(&s_removed[lose_i ? i : j], 1);
    }
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0;
    for (int i = 0; i < nf; ++i)
      if (!s_removed[i]) s_kept[k++] = i;
    s_nk = k;
  }
  __syncthreads();
  const int nk = s_nk;
  if (nk >= 3) {      // remove_outlier, bev/post_parser.py:200-222
    if (tid < nk) {
      const float* ti = cam_trans + (size_t)s_idx[s_kept[tid]] * 3;
      float sum = 0.f, mn = CUDART_INF_F, mx = -CUDART_INF_F;
      for (int j = 0; j < nk; ++j) {
        const float* tj = cam_trans + (size_t)s_idx[s_kept[j]] * 3;
        const float dx = ti[0] - tj[0], dy = ti[1] - tj[1], dz = ti[2] - tj[2];
        const float d = sqrtf(dx * dx + dy * dy + dz * dz);
        sum += d; mn = fminf(mn, d); mx = fmaxf(mx, d);
      }
      s_mean[tid] = (sum - mn - mx) / (float)(nk - 2);       // sorted row without its first and last entry
    }
    __syncthreads();
    if (tid < nk) {
      float tot = 0.f;
      for (int j = 0; j < nk; ++j) tot += s_mean[j];
      const float rel = s_mean[tid] / ((tot - s_mean[tid]) / (float)(nk - 1));
      if (rel > rel_scale_thresh && cam[s_idx[s_kept[tid]] * 3] < scale_thresh) s_removed[s_kept[tid]] = 1;
    }
    __syncthreads();
  }
  if (tid < nf) keep[s_idx[tid]] = s_removed[tid] ? 0 : 1;
}

// ---------------------------------------------------------------------------------------------------------
// Crowd mode (BEV.process_long_image, bev/main.py:184-258).  Crop c of the plan covers padded columns [plan[2c], plan[2c+1]);
// drop_boundary_ratio r_c = (right_c - left_{c+1}) / h / 2 (:213-214, :223-224), evaluated in fp64 like numpy and rounded
// to fp32 for the comparison like torch against a Python scalar.
__device__ __forceinline__ double drop_ratio(const int* plan, int c, int h) {
  return (double)(plan[2 * c + 1] - plan[2 * c + 2]) / (double)h / 2.0;
}

// exclude_boudary_subjects (split2process.py:41-46, tolerance 0): every crop but the last drops cam_x > 1 - r_c
// (bev/main.py:209-215); crop c+1 drops cam_x < r_c - 1 for c in 1..S-2 (:221-226), so crop 1 is never tested on its left.
__global__ void __launch_bounds__(256) bev_long_boundary_kernel(const float* __restrict__ cam, const long long* __restrict__ batch_ids,
                                                                const int* __restrict__ d_count, const int* __restrict__ plan,
                                                                int n_crops, int first_crop, int h, int* __restrict__ valid) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  if (n >= *d_count) return;
  const int c = (int)batch_ids[n] + first_crop;
  const float x = cam[n * 3 + 2];
  bool drop = false;
  if (c != n_crops - 1) drop = x > (float)(1.0 - drop_ratio(plan, c, h) + 0.0);
  if (c >= 2) drop = drop || x < (float)(drop_ratio(plan, c - 1, h) - 1.0 - 0.0);
  valid[n] = drop ? 0 : 1;
}

// convert_crop_cam_params2full_image (split2process.py:48-58) with the crop box shifted by -pad (bev/main.py:247): all three
// components times max(crop w, crop h) / max(h, w), then cam_x += mean(left, right) / (w/2) - 1.  Both factors are fp64
// numpy scalars that torch rounds to fp32; no FMA contraction, like torch's two separate ops.
__global__ void __launch_bounds__(256) bev_long_cam_kernel(const float* __restrict__ cam, const long long* __restrict__ batch_ids,
                                                           const int* __restrict__ d_count, const int* __restrict__ plan, int first_crop,
                                                           int pad, int h, int w, float* __restrict__ cam_full) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  if (n >= *d_count) return;
  const int c = (int)batch_ids[n] + first_crop;
  const int l = plan[2 * c] - pad, r = plan[2 * c + 1] - pad;
  const float sc = (float)((double)max(r - l, h) / (double)max(h, w));
  const float dx = (float)((double)(l + r) / 2.0 / ((double)w / 2.0) - 1.0);
  cam_full[n * 3 + 0] = __fmul_rn(cam[n * 3 + 0], sc);
  cam_full[n * 3 + 1] = __fmul_rn(cam[n * 3 + 1], sc);
  cam_full[n * 3 + 2] = __fadd_rn(__fmul_rn(cam[n * 3 + 2], sc), dx);
}

// survivors of this chunk of crops, in order, appended to the merged buffers: sel / *d_count_sel as bev_compact_kernel,
// *d_base = first merged row of this chunk, *d_merged advanced (clamped to merged_capacity).
__global__ void bev_long_append_kernel(const int* __restrict__ keep, const int* __restrict__ d_count, int merged_capacity,
                                       int* __restrict__ sel, int* __restrict__ d_count_sel, int* __restrict__ d_base,
                                       int* __restrict__ d_merged) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int N = *d_count, base = *d_merged;
  int k = 0;
  for (int i = 0; i < N && base + k < merged_capacity; ++i)
    if (keep[i]) sel[k++] = i;
  *d_count_sel = k;
  *d_base = base;
  *d_merged = base + k;
}

// denormalize_cam_params_to_trans (bev/post_parser.py:114-128), as in bev_unpack_kernel
__global__ void __launch_bounds__(256) bev_cam_trans_kernel(const float* __restrict__ cam, const int* __restrict__ d_count,
                                                            float* __restrict__ cam_trans) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  if (n >= *d_count) return;
  const float depth = 1.f / (cam[n * 3] * kTanFov + 1e-3f);
  cam_trans[n * 3 + 0] = cam[n * 3 + 2] * depth * kTanFov;
  cam_trans[n * 3 + 1] = cam[n * 3 + 1] * depth * kTanFov;
  cam_trans[n * 3 + 2] = depth;
}

// global suppressing_redundant_prediction_via_projection(conf_based=True) (bev/main.py:255) over all merged people: one
// thread per pair (i < j), block row i staged in shared memory; every pair is judged at once, the lower confidence goes.
constexpr int kPairThreads = 128;
__global__ void __launch_bounds__(kPairThreads) bev_long_pairs_kernel(const float* __restrict__ pj2d_org, const float* __restrict__ cam,
                                                                      const float* __restrict__ conf, const int* __restrict__ d_count,
                                                                      float nms_thr_px, int* __restrict__ removed) {
  __shared__ float s_a[142];
  const int i = blockIdx.y, N = *d_count;
  if (i >= N || (int)(blockIdx.x * kPairThreads + kPairThreads - 1) <= i) return;
  for (int k = threadIdx.x; k < 142; k += kPairThreads) s_a[k] = pj2d_org[(size_t)i * 142 + k];
  __syncthreads();
  const int j = blockIdx.x * kPairThreads + threadIdx.x;
  if (j <= i || j >= N) return;
  const float* c = pj2d_org + (size_t)j * 142;
  float sum = 0.f;
  for (int k = 0; k < 71; ++k) {
    const float dx = s_a[2 * k] - c[2 * k], dy = s_a[2 * k + 1] - c[2 * k + 1];
    sum += sqrtf(dx * dx + dy * dy);
  }
  const float si = cam[i * 3] * 2.f, sj = cam[j * 3] * 2.f;
  if (sum / 71.f / fmaxf(si, sj) < nms_thr_px) atomicExch(&removed[conf[i] < conf[j] ? i : j], 1);
}

__global__ void bev_long_kept_kernel(const int* __restrict__ removed, const int* __restrict__ d_count, int* __restrict__ kept,
                                     int* __restrict__ d_nk) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int N = *d_count;
  int k = 0;
  for (int i = 0; i < N; ++i)
    if (!removed[i]) kept[k++] = i;
  *d_nk = k;
}

// remove_outlier row statistic (bev/post_parser.py:206-210) of kept person r: mean of its sorted distance row without
// the first and last entry = (sum - min - max) / (nk - 2)
__global__ void __launch_bounds__(256) bev_long_rowmean_kernel(const float* __restrict__ cam_trans, const int* __restrict__ kept,
                                                               const int* __restrict__ d_nk, float* __restrict__ mean_dist) {
  __shared__ float s_sum[256], s_mn[256], s_mx[256];
  const int r = blockIdx.x, nk = *d_nk, tid = threadIdx.x;
  if (nk < 3 || r >= nk) return;
  const float* ti = cam_trans + (size_t)kept[r] * 3;
  float sum = 0.f, mn = CUDART_INF_F, mx = -CUDART_INF_F;
  for (int j = tid; j < nk; j += 256) {
    const float* tj = cam_trans + (size_t)kept[j] * 3;
    const float dx = ti[0] - tj[0], dy = ti[1] - tj[1], dz = ti[2] - tj[2];
    const float d = sqrtf(dx * dx + dy * dy + dz * dz);
    sum += d; mn = fminf(mn, d); mx = fmaxf(mx, d);
  }
  s_sum[tid] = sum; s_mn[tid] = mn; s_mx[tid] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) {
      s_sum[tid] += s_sum[tid + o]; s_mn[tid] = fminf(s_mn[tid], s_mn[tid + o]); s_mx[tid] = fmaxf(s_mx[tid], s_mx[tid + o]);
    }
    __syncthreads();
  }
  if (tid == 0) mean_dist[r] = (s_sum[0] - s_mn[0] - s_mx[0]) / (float)(nk - 2);
}

// remove_outlier flags (bev/post_parser.py:212-221) over the kept people, then the survivors in order -> sel / *d_count_out
__global__ void __launch_bounds__(1024) bev_long_outlier_kernel(const float* __restrict__ cam, const int* __restrict__ kept,
                                                                const int* __restrict__ d_nk, const float* __restrict__ mean_dist,
                                                                float rel_scale_thresh, float scale_thresh, int* __restrict__ removed,
                                                                const int* __restrict__ d_count, int* __restrict__ sel,
                                                                int* __restrict__ d_count_out) {
  __shared__ float s_red[1024];
  const int nk = *d_nk, tid = threadIdx.x;
  if (nk >= 3) {
    float t = 0.f;
    for (int r = tid; r < nk; r += 1024) t += mean_dist[r];
    s_red[tid] = t;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
      if (tid < o) s_red[tid] += s_red[tid + o];
      __syncthreads();
    }
    const float tot = s_red[0];
    for (int r = tid; r < nk; r += 1024) {
      const float rel = mean_dist[r] / ((tot - mean_dist[r]) / (float)(nk - 1));
      if (rel > rel_scale_thresh && cam[kept[r] * 3] < scale_thresh) removed[kept[r]] = 1;
    }
    __syncthreads();
  }
  if (tid == 0) {
    const int N = *d_count;
    int k = 0;
    for (int i = 0; i < N; ++i)
      if (!removed[i]) sel[k++] = i;
    *d_count_out = k;
  }
}

__global__ void bev_compact_kernel(const int* __restrict__ keep, const int* __restrict__ d_count, int* __restrict__ sel,
                                   int* __restrict__ d_count_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int N = *d_count;
  int k = 0;
  for (int i = 0; i < N; ++i)
    if (keep[i]) sel[k++] = i;
  *d_count_out = k;
}

// d_base (may be NULL): device row offset into dst
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint32_t* __restrict__ src, int row_words, const int* __restrict__ sel,
                                                          const int* __restrict__ d_count, const int* __restrict__ d_base,
                                                          uint32_t* __restrict__ dst) {
  const int i = blockIdx.x;
  if (i >= *d_count) return;
  const uint32_t* s = src + (size_t)sel[i] * row_words;
  uint32_t* d = dst + ((size_t)(d_base ? *d_base : 0) + i) * row_words;
  for (int k = blockIdx.y * 256 + threadIdx.x; k < row_words; k += gridDim.y * 256) d[k] = s[k];
}

}  // namespace b200romp

using namespace b200romp;

struct b200romp_bev {
  int device = 0;
  BevDev dev;
  std::vector<void*> allocs;
};

static const float* up(b200romp_bev* h, const float* host, size_t n, bool* ok) {
  void* d = nullptr;
  if (cudaMalloc(&d, n * sizeof(float)) != cudaSuccess || cudaMemcpy(d, host, n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
    *ok = false;
    return nullptr;
  }
  h->allocs.push_back(d);
  return reinterpret_cast<const float*>(d);
}

extern "C" {

b200romp_bev* b200romp_bev_create(int device, const b200romp_bev_weights* w) {
  if (!w || !w->center_ref || !w->cam_ref || !w->coordmap || !w->anchors || !w->embed || !w->w0 || !w->b0 || !w->w1 || !w->b1 ||
      !w->w2 || !w->b2) {
    set_error("bev_create: null weight pointer");
    return nullptr;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    set_error("bev_create: cudaSetDevice(%d) failed (no CPU fallback)", device);
    return nullptr;
  }
  b200romp_bev* h = new b200romp_bev();
  h->device = device;
  bool ok = true;
  auto transpose = [](const float* src, int rows, int cols) {      // [rows][cols] -> [cols][rows]
    std::vector<float> t((size_t)rows * cols);
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < cols; ++c) t[(size_t)c * rows + r] = src[(size_t)r * cols + c];
    return t;
  };
  BevDev& d = h->dev;
  d.center_ref = up(h, w->center_ref, 56, &ok);
  d.cam_ref = up(h, w->cam_ref, 492, &ok);
  d.coordmap = up(h, w->coordmap, (size_t)kVol * 3, &ok);
  d.anchors = up(h, w->anchors, 64, &ok);
  d.embed = up(h, w->embed, 128 * 128, &ok);
  std::vector<float> t0 = transpose(w->w0, 512, 128), t1 = transpose(w->w1, 512, 512), t2 = transpose(w->w2, 143, 512);
  d.w0t = up(h, t0.data(), t0.size(), &ok); d.b0 = up(h, w->b0, 512, &ok);
  d.w1t = up(h, t1.data(), t1.size(), &ok); d.b1 = up(h, w->b1, 512, &ok);
  d.w2t = up(h, t2.data(), t2.size(), &ok); d.b2 = up(h, w->b2, 143, &ok);
  if (!ok) {
    set_error("bev_create: upload failed (%s)", cudaGetErrorString(cudaGetLastError()));
    b200romp_bev_destroy(h);
    return nullptr;
  }
  return h;
}

void b200romp_bev_destroy(b200romp_bev* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

int b200romp_bev_bv_input(const float* maps_fv, const void* img_feats, int feats_dtype, int feats_C, int batch, void* out, int out_dtype,
                          b200romp_stream stream) {
  B2R_REQUIRE(maps_fv && img_feats && out && batch > 0 && feats_C >= 16, "bev_bv_input: bad arguments");
  const size_t n = (size_t)batch * kS * 2560;
  bev_bv_input_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(maps_fv, img_feats, feats_dtype, feats_C, batch, out, out_dtype);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_bev_center3d(b200romp_bev* h, const float* maps_fv, const void* bv_out, int bv_dtype, int batch, float* tmp,
                          float* center3d, b200romp_stream stream) {
  B2R_REQUIRE(h && maps_fv && bv_out && tmp && center3d && batch > 0, "bev_center3d: bad arguments");
  B2R_CUDA_OK(cudaSetDevice(h->device));
  static const bool two_pass = [] { const char* e = getenv("B200ROMP_BEV_CENTER3D_2PASS"); return e && e[0] == '1'; }();
  if (two_pass) {                      // round-1 formulation (one thread per voxel, intermediate in `tmp`): kept for A/B checks
    const size_t n = (size_t)batch * kVol;
    const unsigned g = (unsigned)((n + 255) / 256);
    bev_center3d_kernel<<<g, 256, 0, (cudaStream_t)stream>>>(maps_fv, bv_out, bv_dtype, h->dev, batch, nullptr, tmp, 1);
    bev_center3d_kernel<<<g, 256, 0, (cudaStream_t)stream>>>(maps_fv, bv_out, bv_dtype, h->dev, batch, tmp, center3d, 2);
  } else {
    dim3 grid((kS / kTW) * (kS / kTH), kD / kTD, batch);
    bev_center3d_fused_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(maps_fv, bv_out, bv_dtype, h->dev, center3d);
  }
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

long long b200romp_bev_parse_workspace_bytes(int batch) {
  return (long long)batch * (sizeof(int) * 2 + kCandCap * 8 + kMaxP * 8);
}

int b200romp_bev_parse3d(const float* center3d, int batch, float thresh, int capacity, int* d_count, long long* batch_ids,
                         long long* czyx, float* conf, void* workspace, b200romp_stream stream_) {
  B2R_REQUIRE(center3d && d_count && batch_ids && czyx && conf && workspace && batch > 0 && capacity > 0, "bev_parse3d: bad arguments");
  B2R_REQUIRE(thresh >= 0.f, "bev_parse3d: thresh must be >= 0");
  cudaStream_t stream = (cudaStream_t)stream_;
  int* cand_count = reinterpret_cast<int*>(workspace);
  int* counts = cand_count + batch;
  int* cand_idx = counts + batch;
  float* cand_val = reinterpret_cast<float*>(cand_idx + (size_t)batch * kCandCap);
  int* top_idx = reinterpret_cast<int*>(cand_val + (size_t)batch * kCandCap);
  float* top_val = reinterpret_cast<float*>(top_idx + (size_t)batch * kMaxP);
  B2R_CUDA_OK(cudaMemsetAsync(cand_count, 0, sizeof(int) * batch, stream));
  const size_t n = (size_t)batch * kVol;
  bev_nms3d_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(center3d, batch, thresh, cand_count, cand_idx, cand_val);
  bev_top64_kernel<<<batch, 1024, 0, stream>>>(cand_count, cand_idx, cand_val, counts, top_idx, top_val);
  bev_emit_kernel<<<batch, 64, 0, stream>>>(batch, capacity, counts, top_idx, top_val, d_count, batch_ids, czyx, conf);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_bev_regress(b200romp_bev* h, const float* maps_fv, const void* bv_out, int bv_dtype, const void* fv_feats, int fv_dtype,
                         int capacity, const int* d_count, const long long* batch_ids, const long long* czyx, float* params_pred,
                         long long* cam_czyx, float* cam, float* thetas, float* betas, float* cam_trans, b200romp_stream stream_) {
  B2R_REQUIRE(h && maps_fv && bv_out && fv_feats && d_count && batch_ids && czyx && params_pred && cam_czyx && cam && thetas &&
                  betas && cam_trans && capacity > 0, "bev_regress: bad arguments");
  B2R_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t stream = (cudaStream_t)stream_;
  bev_regress_kernel<<<capacity, 256, 0, stream>>>(h->dev, maps_fv, bv_out, bv_dtype, fv_feats, fv_dtype, d_count, batch_ids, czyx,
                                                   params_pred, cam_czyx);
  bev_unpack_kernel<<<capacity, 64, 0, stream>>>(params_pred, d_count, cam, thetas, betas, cam_trans);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_bev_post(const float* betas, const float* verts_smil, const float* joints_smil, float* verts, float* joints,
                      const float* cam, const float* cam_trans, const long long* batch_ids, int batch, int capacity,
                      const int* d_count, const float* offsets6, float nms_thresh, float rel_scale_thresh, float img_max_side,
                      float* pj2d_org, int* keep, int* sel, int* d_count_out, b200romp_stream stream_) {
  B2R_REQUIRE(betas && verts && joints && cam && cam_trans && batch_ids && d_count && offsets6 && pj2d_org && keep && sel &&
                  d_count_out && batch > 0 && capacity > 0, "bev_post: bad arguments");
  cudaStream_t stream = (cudaStream_t)stream_;
  if (verts_smil && joints_smil)
    bev_merge_smil_kernel<<<dim3(capacity, 4), 256, 0, stream>>>(betas, d_count, verts_smil, joints_smil, verts, joints);
  const float top = offsets6[0], left = offsets6[2], hh = offsets6[4], ww = offsets6[5];
  bev_project_kernel<<<capacity, 128, 0, stream>>>(joints, cam_trans, d_count, hh > ww ? hh : ww, left, top, pj2d_org);
  B2R_CUDA_OK(cudaMemsetAsync(keep, 0, sizeof(int) * capacity, stream));
  bev_postfilter_kernel<<<batch, 256, 0, stream>>>(pj2d_org, cam, cam_trans, batch_ids, d_count, nms_thresh * img_max_side / 640.f,
                                                   rel_scale_thresh, nullptr, 0.25f, nullptr, keep);
  bev_compact_kernel<<<1, 32, 0, stream>>>(keep, d_count, sel, d_count_out);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_gather_rows(const void* src, int row_bytes, const int* sel, const int* d_count, int capacity, void* dst,
                         b200romp_stream stream) {
  return b200romp_gather_rows_at(src, row_bytes, sel, d_count, nullptr, capacity, dst, stream);
}

int b200romp_gather_rows_at(const void* src, int row_bytes, const int* sel, const int* d_count, const int* d_base, int capacity,
                            void* dst, b200romp_stream stream) {
  B2R_REQUIRE(src && sel && d_count && dst && row_bytes > 0 && row_bytes % 4 == 0 && capacity > 0, "gather_rows: bad arguments");
  const int words = row_bytes / 4;
  gather_rows_kernel<<<dim3(capacity, words > 4096 ? 8 : 1), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint32_t*>(src), words, sel, d_count, d_base, reinterpret_cast<uint32_t*>(dst));
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_bev_long_crops(const float* betas, const float* verts_smil, const float* joints_smil, float* verts, float* joints,
                            const float* cam, const float* cam_trans, const float* conf, const long long* batch_ids, int batch,
                            int capacity, const int* d_count, const int* plan, int n_crops, int first_crop, int h, int w, int pad,
                            float crop_nms_thr_px, float rel_scale_thresh, float* pj2d_org, float* cam_full, int* flags, int* sel,
                            int* d_count_sel, int* d_base, int* d_merged, int merged_capacity, b200romp_stream stream_) {
  B2R_REQUIRE(betas && verts && joints && cam && cam_trans && conf && batch_ids && d_count && plan && pj2d_org && cam_full && flags &&
                  sel && d_count_sel && d_base && d_merged && batch > 0 && capacity > 0 && n_crops >= 2 && first_crop >= 0 &&
                  first_crop + batch <= n_crops && h > 0 && w > 0 && pad >= 0 && merged_capacity > 0,
              "bev_long_crops: bad arguments");
  cudaStream_t stream = (cudaStream_t)stream_;
  int *valid = flags, *keep = flags + capacity;
  const unsigned g = (unsigned)((capacity + 255) / 256);
  if (verts_smil && joints_smil)
    bev_merge_smil_kernel<<<dim3(capacity, 4), 256, 0, stream>>>(betas, d_count, verts_smil, joints_smil, verts, joints);
  bev_long_boundary_kernel<<<g, 256, 0, stream>>>(cam, batch_ids, d_count, plan, n_crops, first_crop, h, valid);
  // crop pixels: input2org_offsets [0, ch, 0, cw, ch, cw] (bev/main.py:216-217); the crop width never exceeds h
  bev_project_kernel<<<capacity, 128, 0, stream>>>(joints, cam_trans, d_count, (float)h, 0.f, 0.f, pj2d_org);
  B2R_CUDA_OK(cudaMemsetAsync(keep, 0, sizeof(int) * capacity, stream));
  bev_postfilter_kernel<<<batch, 256, 0, stream>>>(pj2d_org, cam, cam_trans, batch_ids, d_count, crop_nms_thr_px, rel_scale_thresh,
                                                   conf, 1.f, valid, keep);                   // :228-232
  bev_long_cam_kernel<<<g, 256, 0, stream>>>(cam, batch_ids, d_count, plan, first_crop, pad, h, w, cam_full);
  bev_long_append_kernel<<<1, 32, 0, stream>>>(keep, d_count, merged_capacity, sel, d_count_sel, d_base, d_merged);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

int b200romp_bev_long_merge(const float* joints, const float* cam, const float* conf, int capacity, const int* d_count, int h, int w,
                            float nms_thr_px, float rel_scale_thresh, float* cam_trans, float* pj2d_org, int* workspace, int* sel,
                            int* d_count_out, b200romp_stream stream_) {
  B2R_REQUIRE(joints && cam && conf && d_count && cam_trans && pj2d_org && workspace && sel && d_count_out && capacity > 0 && h > 0 &&
                  w > 0, "bev_long_merge: bad arguments");
  B2R_REQUIRE(capacity <= 65535, "bev_long_merge: capacity > 65535");
  cudaStream_t stream = (cudaStream_t)stream_;
  int *removed = workspace, *kept = workspace + capacity, *d_nk = workspace + 2 * capacity;
  float* mean_dist = reinterpret_cast<float*>(workspace + 2 * capacity + 1);
  const unsigned g = (unsigned)((capacity + 255) / 256);
  const int side = h > w ? h : w;
  bev_cam_trans_kernel<<<g, 256, 0, stream>>>(cam, d_count, cam_trans);                       // bev/main.py:253
  bev_project_kernel<<<capacity, 128, 0, stream>>>(joints, cam_trans, d_count, (float)side, 0.f, (float)((w - h) / 2), pj2d_org);
  B2R_CUDA_OK(cudaMemsetAsync(removed, 0, sizeof(int) * capacity, stream));
  bev_long_pairs_kernel<<<dim3((capacity + kPairThreads - 1) / kPairThreads, capacity), kPairThreads, 0, stream>>>(
      pj2d_org, cam, conf, d_count, nms_thr_px, removed);                                     // :255
  bev_long_kept_kernel<<<1, 32, 0, stream>>>(removed, d_count, kept, d_nk);
  bev_long_rowmean_kernel<<<capacity, 256, 0, stream>>>(cam_trans, kept, d_nk, mean_dist);     // :256
  bev_long_outlier_kernel<<<1, 1024, 0, stream>>>(cam, kept, d_nk, mean_dist, rel_scale_thresh, 0.5f, removed, d_count, sel,
                                                  d_count_out);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

}  // extern "C"
