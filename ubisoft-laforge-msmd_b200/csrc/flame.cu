// FLAME decode: pack + per-frame pose/chain kernel + CUDA-core fused blendshape/LBS kernel.
//
// Replaces utils/flame.py:180-244 (FLAME.forward) and utils/lbs.py:141-371 (lbs, blend_shapes,
// vertices2joints, batch_rodrigues, batch_rigid_transform).  The reference materialises
// v_shaped, pose_offsets, the per-vertex 4x4 T ([B,V,16] = 2.6 GB at B=8192) and v_homo; here
// one GEMM over K = NB + 36 produces v_posed - template tile by tile and the skinning is its
// epilogue, so HBM sees only betas/pose in and vertices out.
#include "flame.cuh"
#include <cmath>
#include "rot_math.cuh"
#include "profile.cuh"
#include <vector>
#include <cstring>
#include <cstdlib>

namespace msmd {

// ---------------------------------------------------------------------------------------
// Per-frame kernel: one warp per frame.
//   A[b] = betas[b] | vec(R[1:] - I) | 0          (lbs.py:200-201 pose_feature)
//   J[b] = Jt + Jb @ betas[b]                     (lbs.py:189 with the regressor folded)
//   chain (lbs.py:317-371) -> xf[b][j] = G_j (9) | t_j - G_j J_j (3)
// ---------------------------------------------------------------------------------------
template <int NJ>
__global__ void __launch_bounds__(256, 3) flame_pose_kernel(const float* __restrict__ betas, const float* __restrict__ pose,
                                                         int pose2rot, int64_t B, int NB, int Kpad,
                                                         const float* __restrict__ Jt, const float* __restrict__ Jb,
                                                         const int* __restrict__ parents_g, float* __restrict__ A,
                                                         __half* __restrict__ A_hi, __half* __restrict__ A_lo,
                                                         float* __restrict__ xf, float* __restrict__ joints_out) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const float* be = betas + b * NB;
  float* Arow = A + b * Kpad;
  float acc[NJ * 3];
#pragma unroll
  for (int i = 0; i < NJ * 3; ++i) acc[i] = 0.f;
  // every coefficient of the frame is requested before the first one is used (NB <= 512: 16 per lane); the loop used to
  // pay one memory latency per 32 coefficients (ncu: 70% of the kernel's stall samples on the first use of be[k])
  constexpr int kMaxIt = 16;
  float bv[kMaxIt];
#pragma unroll
  for (int it = 0; it < kMaxIt; ++it) {
    const int k = lane + 32 * it;
    bv[it] = k < NB ? be[k] : 0.f;
  }
#pragma unroll
  for (int it = 0; it < kMaxIt; ++it) {
    const int k = lane + 32 * it;
    if (k < NB) {
      const float v = bv[it];
      if (A_hi == nullptr) Arow[k] = v;      // the fp32 copy is only read by the CUDA-core path (impl 1)
      if (A_hi) {
        const float sv = v * kFlameScaleA;
        const __half hi = __float2half_rn(sv);
        A_hi[b * Kpad + k] = hi;
        A_lo[b * Kpad + k] = __float2half_rn(sv - __half2float(hi));
      }
#pragma unroll
      for (int i = 0; i < NJ * 3; ++i) acc[i] = fmaf(__ldg(Jb + i * NB + k), v, acc[i]);
    }
  }
  for (int k = lane + 32 * kMaxIt; k < NB; k += 32) {   // NB > 512 (not a FLAME model): plain loop
    const float v = be[k];
    if (A_hi == nullptr) Arow[k] = v;
    if (A_hi) {
      const float sv = v * kFlameScaleA;
      const __half hi = __float2half_rn(sv);
      A_hi[b * Kpad + k] = hi;
      A_lo[b * Kpad + k] = __float2half_rn(sv - __half2float(hi));
    }
#pragma unroll
    for (int i = 0; i < NJ * 3; ++i) acc[i] = fmaf(__ldg(Jb + i * NB + k), v, acc[i]);
  }
#pragma unroll
  for (int i = 0; i < NJ * 3; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  }
  const int K = NB + (NJ - 1) * 9;
  for (int k = K + lane; k < Kpad; k += 32) {
    if (A_hi == nullptr) Arow[k] = 0.f;
    if (A_hi) { A_hi[b * Kpad + k] = __float2half_rn(0.f); A_lo[b * Kpad + k] = __float2half_rn(0.f); }
  }
  // ---- per-joint work: lane j owns joint j (Rodrigues, pose feature, its link of the kinematic chain); the parent's
  // transform travels by shuffle.  (One lane used to do all five joints serially with the chain's arrays in local
  // memory - `parents` is runtime data - and 130 scalar stores: 53 us per 8192 frames, 14% of the FLAME step.)
  float Jx = 0.f, Jy = 0.f, Jz = 0.f;
#pragma unroll
  for (int j = 0; j < NJ; ++j)
    if (lane == j) { Jx = Jt[j * 3 + 0] + acc[j * 3 + 0]; Jy = Jt[j * 3 + 1] + acc[j * 3 + 1]; Jz = Jt[j * 3 + 2] + acc[j * 3 + 2]; }
  Mat3 Rj;
#pragma unroll
  for (int i = 0; i < 9; ++i) Rj.m[i] = (i % 4 == 0) ? 1.0f : 0.0f;
  if (lane < NJ) {
    if (pose2rot) {
      const float* p = pose + b * NJ * 3 + lane * 3;
      Rj = rodrigues(p[0], p[1], p[2]);
    } else {
      const float* p = pose + b * NJ * 9 + lane * 9;
#pragma unroll
      for (int i = 0; i < 9; ++i) Rj.m[i] = p[i];
    }
  }
  if (lane >= 1 && lane < NJ) {
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float v = Rj.m[i] - ((i % 4 == 0) ? 1.0f : 0.0f);
      const int k = NB + (lane - 1) * 9 + i;
      if (A_hi == nullptr) Arow[k] = v;
      if (A_hi) {
        const float sv = v * kFlameScaleA;
        const __half hi = __float2half_rn(sv);
        A_hi[b * Kpad + k] = hi;
        A_lo[b * Kpad + k] = __float2half_rn(sv - __half2float(hi));
      }
    }
  }
  // chain (lbs.py:317-371): G_j = G_parent R_j, t_j = G_parent (J_j - J_parent) + t_parent; parents[j] < j
  Mat3 G = Rj;
  float tx = Jx, ty = Jy, tz = Jz;
#pragma unroll
  for (int j = 1; j < NJ; ++j) {
    const int pj = parents_g[j];
    Mat3 Gp;
#pragma unroll
    for (int i = 0; i < 9; ++i) Gp.m[i] = __shfl_sync(0xffffffffu, G.m[i], pj);
    const float tpx = __shfl_sync(0xffffffffu, tx, pj), tpy = __shfl_sync(0xffffffffu, ty, pj), tpz = __shfl_sync(0xffffffffu, tz, pj);
    const float Jpx = __shfl_sync(0xffffffffu, Jx, pj), Jpy = __shfl_sync(0xffffffffu, Jy, pj), Jpz = __shfl_sync(0xffffffffu, Jz, pj);
    if (lane == j) {
      const float rx = Jx - Jpx, ry = Jy - Jpy, rz = Jz - Jpz;
      G = mat3_mul(Gp, Rj);
      tx = Gp.m[0] * rx + Gp.m[1] * ry + Gp.m[2] * rz + tpx;
      ty = Gp.m[3] * rx + Gp.m[4] * ry + Gp.m[5] * rz + tpy;
      tz = Gp.m[6] * rx + Gp.m[7] * ry + Gp.m[8] * rz + tpz;
    }
  }
  if (lane < NJ) {
    float* x = xf + b * NJ * 12 + lane * 12;
#pragma unroll
    for (int i = 0; i < 9; ++i) x[i] = G.m[i];
    x[9] = tx - (G.m[0] * Jx + G.m[1] * Jy + G.m[2] * Jz);
    x[10] = ty - (G.m[3] * Jx + G.m[4] * Jy + G.m[5] * Jz);
    x[11] = tz - (G.m[6] * Jx + G.m[7] * Jy + G.m[8] * Jz);
    if (joints_out) {
      joints_out[b * NJ * 3 + lane * 3 + 0] = tx;
      joints_out[b * NJ * 3 + lane * 3 + 1] = ty;
      joints_out[b * NJ * 3 + lane * 3 + 2] = tz;
    }
  }
}

// ---------------------------------------------------------------------------------------
// The same per-frame work with the joint regression on the tensor cores: J = Jt + Jb beta is a [15 x NB] x [NB x frames]
// product, and the one-warp-per-frame kernel above spends ~2500 instructions per frame on it (15 loads + 15 FMAs per
// coefficient and lane).  Here a warp owns 8 frames = the N columns of mma.sync m16n8k16: the rows are the 15 joint
// coordinates, fp16 two-term splits of both operands (three passes, 22 mantissa bits; the split of 16 beta is the very
// operand row the blendshape GEMM needs, so it is produced once and used twice).  The per-joint section then runs on
// lane 8 g + j.  Two warps share 8 frames (half of K each, then 4 frames each).  Needs NJ * 3 <= 16 and an even NB.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void pose_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  const __half2 h = __halves2half2(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
template <int NJ>
__global__ void __launch_bounds__(256) flame_pose_mma_kernel(const float* __restrict__ betas, const float* __restrict__ pose,
                                                             int pose2rot, int64_t B, int NB, int KB, int Kpad,
                                                             const float* __restrict__ Jt, const __half* __restrict__ Jb16,
                                                             const int* __restrict__ parents_g, float* __restrict__ A,
                                                             __half* __restrict__ A_hi, __half* __restrict__ A_lo,
                                                             float* __restrict__ xf, float* __restrict__ joints_out) {
  static_assert(NJ * 3 <= 16 && NJ <= 8, "one 16-row MMA tile of joint coordinates; 8 lanes per frame in the joint section");
  // warps w and w + 4 share 8 frames: each takes half of the K range (the 25 k-steps of one warp were a 30 us dependent
  // chain at 7 warps per SM) and, afterwards, 4 of the 8 frames of the per-joint section
  __shared__ float Jp[2][4][8][16];              // [K half][frame group][frame][joint coordinate] raw partial sums
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
  const int wq = warp & 3, kh = warp >> 2;
  const int64_t f0 = ((int64_t)blockIdx.x * 4 + wq) * 8;
  if (f0 >= B) return;                           // (both warps of the pair leave together; the pair barrier below is theirs alone)
  auto put = [&](int64_t b, int k, float v) {    // one element of the GEMM operand row: fp32 (impl 1) or the fp16 split (impl 0)
    if (A_hi == nullptr) { A[b * Kpad + k] = v; return; }
    const float sv = v * kFlameScaleA;
    const __half hi = __float2half_rn(sv);
    A_hi[b * Kpad + k] = hi;
    A_lo[b * Kpad + k] = __float2half_rn(sv - __half2float(hi));
  };
  // ---- joint regression + operand split of the coefficients
  {
    const int64_t f = f0 + gid;
    const bool fv = f < B;
    const float* be = betas + f * NB;
    const __half* JH = Jb16;
    const __half* JL = Jb16 + 16 * KB;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const int nks = KB / 16, ks_mid = (nks + 1) / 2;
    const int ks_lo = kh == 0 ? 0 : ks_mid, ks_hi = kh == 0 ? ks_mid : nks;
#pragma unroll 4
    for (int ks = ks_lo; ks < ks_hi; ++ks) {
      const int k0 = ks * 16;
      const int ka = k0 + 2 * tig, kb = ka + 8;                 // even: a pair never straddles NB (NB is even)
      float2 xa = make_float2(0.f, 0.f), xb = make_float2(0.f, 0.f);
      if (fv && ka < NB) xa = *reinterpret_cast<const float2*>(be + ka);
      if (fv && kb < NB) xb = *reinterpret_cast<const float2*>(be + kb);
      uint32_t ah[4], al[4];
      ah[0] = __ldg(reinterpret_cast<const uint32_t*>(JH + gid * KB + ka));
      ah[1] = __ldg(reinterpret_cast<const uint32_t*>(JH + (gid + 8) * KB + ka));
      ah[2] = __ldg(reinterpret_cast<const uint32_t*>(JH + gid * KB + kb));
      ah[3] = __ldg(reinterpret_cast<const uint32_t*>(JH + (gid + 8) * KB + kb));
      al[0] = __ldg(reinterpret_cast<const uint32_t*>(JL + gid * KB + ka));
      al[1] = __ldg(reinterpret_cast<const uint32_t*>(JL + (gid + 8) * KB + ka));
      al[2] = __ldg(reinterpret_cast<const uint32_t*>(JL + gid * KB + kb));
      al[3] = __ldg(reinterpret_cast<const uint32_t*>(JL + (gid + 8) * KB + kb));
      const float s0 = xa.x * kFlameScaleA, s1 = xa.y * kFlameScaleA, s2 = xb.x * kFlameScaleA, s3 = xb.y * kFlameScaleA;
      const __half h0 = __float2half_rn(s0), h1 = __float2half_rn(s1), h2 = __float2half_rn(s2), h3 = __float2half_rn(s3);
      const uint32_t bh0 = pack_h2(h0, h1), bh1 = pack_h2(h2, h3);
      const uint32_t bl0 = pack_h2(__float2half_rn(s0 - __half2float(h0)), __float2half_rn(s1 - __half2float(h1)));
      const uint32_t bl1 = pack_h2(__float2half_rn(s2 - __half2float(h2)), __float2half_rn(s3 - __half2float(h3)));
      if (fv) {
        if (A_hi != nullptr) {
          if (ka < NB) { *reinterpret_cast<uint32_t*>(A_hi + f * Kpad + ka) = bh0; *reinterpret_cast<uint32_t*>(A_lo + f * Kpad + ka) = bl0; }
          if (kb < NB) { *reinterpret_cast<uint32_t*>(A_hi + f * Kpad + kb) = bh1; *reinterpret_cast<uint32_t*>(A_lo + f * Kpad + kb) = bl1; }
        } else {
          if (ka < NB) *reinterpret_cast<float2*>(A + f * Kpad + ka) = xa;
          if (kb < NB) *reinterpret_cast<float2*>(A + f * Kpad + kb) = xb;
        }
      }
      pose_mma(acc, al, bh0, bh1);     // lo * hi
      pose_mma(acc, ah, bl0, bl1);     // hi * lo
      pose_mma(acc, ah, bh0, bh1);     // hi * hi
    }
    // partial accumulator (row = joint coordinate, column = frame of the group) -> shared memory
    Jp[kh][wq][2 * tig][gid] = acc[0];
    Jp[kh][wq][2 * tig + 1][gid] = acc[1];
    Jp[kh][wq][2 * tig][gid + 8] = acc[2];
    Jp[kh][wq][2 * tig + 1][gid + 8] = acc[3];
  }
  asm volatile("bar.sync %0, 64;" ::"r"(1 + wq) : "memory");     // the two warps of this frame group
  const int K = NB + (NJ - 1) * 9;
  for (int fs = kh; fs < 8; fs += 2) {
    if (f0 + fs < B)
      for (int k = K + lane; k < Kpad; k += 32) put(f0 + fs, k, 0.f);
  }
  // ---- per-joint section: this warp takes frames 4 kh .. 4 kh + 3 of the group; lane 8 g + j owns joint j of frame 4 kh + g
  {
    constexpr float kInv = 1.0f / (kFlameScaleA * kFlameScaleJ);
    const int fs = 4 * kh + (lane >> 3), jn = lane & 7;
    const int64_t b = f0 + fs;
    const bool mine = jn < NJ && b < B;
    float Jx = 0.f, Jy = 0.f, Jz = 0.f;
    if (jn < NJ) {      // J = Jt + (K half 0 + K half 1) / scale, in that order
      Jx = fmaf(Jp[0][wq][fs][3 * jn] + Jp[1][wq][fs][3 * jn], kInv, Jt[3 * jn]);
      Jy = fmaf(Jp[0][wq][fs][3 * jn + 1] + Jp[1][wq][fs][3 * jn + 1], kInv, Jt[3 * jn + 1]);
      Jz = fmaf(Jp[0][wq][fs][3 * jn + 2] + Jp[1][wq][fs][3 * jn + 2], kInv, Jt[3 * jn + 2]);
    }
    Mat3 Rj;
#pragma unroll
    for (int i = 0; i < 9; ++i) Rj.m[i] = (i % 4 == 0) ? 1.0f : 0.0f;
    if (mine) {
      if (pose2rot) {
        const float* p = pose + b * NJ * 3 + jn * 3;
        Rj = rodrigues(p[0], p[1], p[2]);
      } else {
        const float* p = pose + b * NJ * 9 + jn * 9;
#pragma unroll
        for (int i = 0; i < 9; ++i) Rj.m[i] = p[i];
      }
    }
    if (mine && jn >= 1) {
#pragma unroll
      for (int i = 0; i < 9; ++i) put(b, NB + (jn - 1) * 9 + i, Rj.m[i] - ((i % 4 == 0) ? 1.0f : 0.0f));
    }
    // chain (lbs.py:317-371): G_j = G_parent R_j, t_j = G_parent (J_j - J_parent) + t_parent; parents[j] < j
    Mat3 G = Rj;
    float tx = Jx, ty = Jy, tz = Jz;
#pragma unroll
    for (int j = 1; j < NJ; ++j) {
      const int src = (lane & 24) | parents_g[j];     // the parent's lane in this lane's frame group
      Mat3 Gp;
#pragma unroll
      for (int i = 0; i < 9; ++i) Gp.m[i] = __shfl_sync(0xffffffffu, G.m[i], src);
      const float tpx = __shfl_sync(0xffffffffu, tx, src), tpy = __shfl_sync(0xffffffffu, ty, src), tpz = __shfl_sync(0xffffffffu, tz, src);
      const float Jpx = __shfl_sync(0xffffffffu, Jx, src), Jpy = __shfl_sync(0xffffffffu, Jy, src), Jpz = __shfl_sync(0xffffffffu, Jz, src);
      if (jn == j) {
        const float rx = Jx - Jpx, ry = Jy - Jpy, rz = Jz - Jpz;
        G = mat3_mul(Gp, Rj);
        tx = Gp.m[0] * rx + Gp.m[1] * ry + Gp.m[2] * rz + tpx;
        ty = Gp.m[3] * rx + Gp.m[4] * ry + Gp.m[5] * rz + tpy;
        tz = Gp.m[6] * rx + Gp.m[7] * ry + Gp.m[8] * rz + tpz;
      }
    }
    if (mine) {
      float* x = xf + b * NJ * 12 + jn * 12;
#pragma unroll
      for (int i = 0; i < 9; ++i) x[i] = G.m[i];
      x[9] = tx - (G.m[0] * Jx + G.m[1] * Jy + G.m[2] * Jz);
      x[10] = ty - (G.m[3] * Jx + G.m[4] * Jy + G.m[5] * Jz);
      x[11] = tz - (G.m[6] * Jx + G.m[7] * Jy + G.m[8] * Jz);
      if (joints_out) {
        joints_out[b * NJ * 3 + jn * 3 + 0] = tx;
        joints_out[b * NJ * 3 + jn * 3 + 1] = ty;
        joints_out[b * NJ * 3 + jn * 3 + 2] = tz;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// CUDA-core fused kernel (impl=1; also the cross-check of the tensor-core path).
// Tile: 64 frames x 96 columns (32 vertices), BK=16, 256 threads, 4x6 register tile.
// ---------------------------------------------------------------------------------------
constexpr int FBM = 64, FBN = 96, FBK = 16;

template <int NJ>
__global__ void __launch_bounds__(256) flame_simt_kernel(const float* __restrict__ A, const float* __restrict__ basis,
                                                         const float* __restrict__ tmpl, const float* __restrict__ W,
                                                         const float* __restrict__ xf, int64_t B, int V, int Kpad,
                                                         float* __restrict__ out) {
  __shared__ float As[FBK][FBM + 4];
  __shared__ float Bs[FBK][FBN + 4];
  __shared__ float sXf[FBM][NJ * 12 + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // tx: vertex pair, ty: frame quad
  const int64_t row0 = (int64_t)blockIdx.y * FBM;
  const int col0 = blockIdx.x * FBN;
  const int N3 = 3 * V;

  for (int i = tid; i < FBM * NJ * 12; i += 256) {
    const int r = i / (NJ * 12), c = i % (NJ * 12);
    const int64_t rr = min(row0 + r, B - 1);
    sXf[r][c] = xf[rr * NJ * 12 + c];
  }

  float acc[4][6];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < Kpad; k0 += FBK) {
    {  // A tile: 64 rows x 16 k = 256 float4
      const int r = tid >> 2, q = tid & 3;
      const int64_t rr = min(row0 + r, B - 1);
      const float4 v = *reinterpret_cast<const float4*>(A + rr * Kpad + k0 + q * 4);
      As[q * 4 + 0][r] = v.x; As[q * 4 + 1][r] = v.y; As[q * 4 + 2][r] = v.z; As[q * 4 + 3][r] = v.w;
    }
    for (int i = tid; i < FBN * 4; i += 256) {  // basis tile: 96 rows x 16 k = 384 float4 (rows padded to N3pad)
      const int r = i >> 2, q = i & 3;
      const float4 v = *reinterpret_cast<const float4*>(basis + (int64_t)(col0 + r) * Kpad + k0 + q * 4);
      Bs[q * 4 + 0][r] = v.x; Bs[q * 4 + 1][r] = v.y; Bs[q * 4 + 2][r] = v.z; Bs[q * 4 + 3][r] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < FBK; ++k) {
      float a[4], bb[6];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 6; ++j) bb[j] = Bs[k][tx * 6 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }

  // Epilogue: v_posed = acc + template; blend the NJ affines with W[v]; apply (lbs.py:210-221).
#pragma unroll
  for (int vv = 0; vv < 2; ++vv) {
    const int n0 = col0 + tx * 6 + vv * 3;
    const int v = n0 / 3;
    if (n0 >= N3) continue;
    float w[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) w[j] = W[v * NJ + j];
    const float t0 = tmpl[n0], t1 = tmpl[n0 + 1], t2 = tmpl[n0 + 2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty * 4 + i;
      if (row0 + r >= B) continue;
      float T[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) s = fmaf(w[j], sXf[r][j * 12 + e], s);
        T[e] = s;
      }
      const float px = acc[i][vv * 3 + 0] + t0, py = acc[i][vv * 3 + 1] + t1, pz = acc[i][vv * 3 + 2] + t2;
      float* o = out + (row0 + r) * N3 + n0;
      o[0] = T[0] * px + T[1] * py + T[2] * pz + T[9];
      o[1] = T[3] * px + T[4] * py + T[5] * pz + T[10];
      o[2] = T[6] * px + T[7] * py + T[8] * pz + T[11];
    }
  }
}

// utils/lbs.py:102-138 vertices2landmarks: one thread per (b, l, xyz)
__global__ void landmarks_kernel(const float* __restrict__ verts, const int64_t* __restrict__ faces,
                                 const int64_t* __restrict__ idx, const float* __restrict__ bary, int64_t B, int V,
                                 int L, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * L * 3) return;
  const int c = (int)(i % 3);
  const int64_t bl = i / 3;
  const int64_t b = bl / L;
  const int64_t f = idx[bl];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) s += verts[(b * V + faces[f * 3 + k]) * 3 + c] * bary[bl * 3 + k];
  out[i] = s;
}

// utils/flame.py:126-172 (_find_dynamic_lmk_idx_and_bcoords) + utils/lbs.py:26-32 (rot_mat_to_euler):
// compose the neck kinematic chain, take the yaw in whole degrees (round-half-even, clamp 39) and map
// it to a row of the 79-entry contour table.
__global__ void contour_index_kernel(const float* __restrict__ pose, int pose2rot, int NJ,
                                     const int64_t* __restrict__ chain, int n_chain, int64_t B,
                                     int64_t* __restrict__ out) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Mat3 rel = {{1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f}};
  for (int i = 0; i < n_chain; ++i) {
    const int j = (int)chain[i];
    Mat3 R;
    if (pose2rot) {
      const float* p = pose + (b * NJ + j) * 3;
      R = rodrigues(p[0], p[1], p[2]);
    } else {
      const float* p = pose + (b * NJ + j) * 9;
      for (int k = 0; k < 9; ++k) R.m[k] = p[k];
    }
    rel = mat3_mul(R, rel);
  }
  const float sy = sqrtf(rel.m[0] * rel.m[0] + rel.m[3] * rel.m[3]);
  const float ang = atan2f(-rel.m[6], sy) * 180.0f / 3.14159265358979323846f;
  long long y = (long long)rintf(fminf(ang, 39.0f));
  if (y < 0) y = (y < -39) ? 78 : (39 - y);
  out[b] = y;
}

static int ensure_workspace(msmd_flame* fh, int64_t B) {
  if (B <= fh->cap_B) return MSMD_OK;
  cudaFree(fh->A); cudaFree(fh->A_hi); cudaFree(fh->A_lo); cudaFree(fh->xf);
  fh->A = fh->xf = nullptr;
  fh->A_hi = fh->A_lo = nullptr;
  fh->cap_B = 0;
  const int64_t cap = ((B + 127) / 128) * 128;  // whole 128-frame tiles for the TMA path
  MSMD_CHECK_CUDA(cudaMalloc(&fh->A, cap * fh->Kpad * sizeof(float)));
  MSMD_CHECK_CUDA(cudaMalloc(&fh->A_hi, cap * fh->Kpad * sizeof(__half)));
  MSMD_CHECK_CUDA(cudaMalloc(&fh->A_lo, cap * fh->Kpad * sizeof(__half)));
  MSMD_CHECK_CUDA(cudaMalloc(&fh->xf, cap * fh->NJ * 12 * sizeof(float)));
  MSMD_CHECK_CUDA(cudaMemset(fh->A, 0, cap * fh->Kpad * sizeof(float)));
  MSMD_CHECK_CUDA(cudaMemset(fh->A_hi, 0, cap * fh->Kpad * sizeof(__half)));
  MSMD_CHECK_CUDA(cudaMemset(fh->A_lo, 0, cap * fh->Kpad * sizeof(__half)));
  MSMD_CHECK_CUDA(cudaMemset(fh->xf, 0, cap * fh->NJ * 12 * sizeof(float)));
  fh->cap_B = cap;
  return MSMD_OK;
}

}  // namespace msmd

using namespace msmd;

extern "C" int msmd_flame_create(const float* v_template, const float* shapedirs, const float* posedirs,
                                 const float* J_regressor, const int64_t* parents, const float* lbs_weights, int V,
                                 int NB, int NJ, int device, msmd_flame** out) {
  MSMD_REQUIRE(out, "msmd_flame_create: null out");
  MSMD_REQUIRE(v_template && shapedirs && posedirs && J_regressor && parents && lbs_weights,
               "msmd_flame_create: null asset pointer");
  MSMD_REQUIRE(V > 0 && NB > 0, "msmd_flame_create: bad sizes V=%d NB=%d", V, NB);
  if (NJ != 5) {
    set_error("msmd_flame_create: only the 5-joint FLAME kinematic tree is supported (got %d)", NJ);
    return MSMD_ERR_UNSUPPORTED;
  }
  MSMD_CHECK_CUDA(cudaSetDevice(device));
  const int P = (NJ - 1) * 9;
  const int N3 = 3 * V, K = NB + P;
  const int Kpad = (K + 63) / 64 * 64;
  const int N3pad = (N3 + 383) / 384 * 384;
  // Stage the assets on the host (they may live on either side); packing is a one-off.
  std::vector<float> h_t(N3), h_s((size_t)N3 * NB), h_p((size_t)P * N3), h_j((size_t)NJ * V), h_w((size_t)V * NJ);
  std::vector<int64_t> h_par(NJ);
  MSMD_CHECK_CUDA(cudaMemcpy(h_t.data(), v_template, h_t.size() * 4, cudaMemcpyDefault));
  MSMD_CHECK_CUDA(cudaMemcpy(h_s.data(), shapedirs, h_s.size() * 4, cudaMemcpyDefault));
  MSMD_CHECK_CUDA(cudaMemcpy(h_p.data(), posedirs, h_p.size() * 4, cudaMemcpyDefault));
  MSMD_CHECK_CUDA(cudaMemcpy(h_j.data(), J_regressor, h_j.size() * 4, cudaMemcpyDefault));
  MSMD_CHECK_CUDA(cudaMemcpy(h_w.data(), lbs_weights, h_w.size() * 4, cudaMemcpyDefault));
  MSMD_CHECK_CUDA(cudaMemcpy(h_par.data(), parents, NJ * 8, cudaMemcpyDefault));
  for (int j = 1; j < NJ; ++j)
    MSMD_REQUIRE(h_par[j] >= 0 && h_par[j] < j, "msmd_flame_create: parents[%d]=%lld is not an earlier joint", j,
                 (long long)h_par[j]);

  msmd_flame* fh = new msmd_flame();
  fh->device = device; fh->V = V; fh->NB = NB; fh->NJ = NJ; fh->N3 = N3; fh->K = K; fh->Kpad = Kpad; fh->N3pad = N3pad;
  fh->parents[0] = -1;
  for (int j = 1; j < NJ; ++j) fh->parents[j] = (int)h_par[j];

  std::vector<float> basis((size_t)N3pad * Kpad, 0.f);
  std::vector<__half> hi(basis.size()), lo(basis.size());
  for (int n = 0; n < N3; ++n) {
    float* row = basis.data() + (size_t)n * Kpad;
    memcpy(row, h_s.data() + (size_t)n * NB, NB * sizeof(float));
    for (int p = 0; p < P; ++p) row[NB + p] = h_p[(size_t)p * N3 + n];
  }
  for (size_t i = 0; i < basis.size(); ++i) {
    const float sv = basis[i] * kFlameScaleB;
    if (!(fabsf(sv) < 60000.0f)) {   // |entry| >= 234: not a blendshape basis in metres (and it would overflow the fp16 split)
      delete fh;
      set_error("msmd_flame_create: blendshape basis entry %g is outside the range of the fp16 two-term split (|x| < 234)", basis[i]);
      return MSMD_ERR_INVALID;
    }
    hi[i] = __float2half_rn(sv);
    lo[i] = __float2half_rn(sv - __half2float(hi[i]));
  }
  // Joint regression folded through the blendshapes (double accumulation on the host).
  std::vector<float> Jt(NJ * 3), Jb((size_t)NJ * 3 * NB);
  for (int j = 0; j < NJ; ++j)
    for (int c = 0; c < 3; ++c) {
      double s = 0;
      for (int v = 0; v < V; ++v) s += (double)h_j[(size_t)j * V + v] * h_t[(size_t)v * 3 + c];
      Jt[j * 3 + c] = (float)s;
      for (int l = 0; l < NB; ++l) {
        double a = 0;
        for (int v = 0; v < V; ++v) a += (double)h_j[(size_t)j * V + v] * h_s[((size_t)v * 3 + c) * NB + l];
        Jb[(size_t)(j * 3 + c) * NB + l] = (float)a;
      }
    }
  // fp16 two-term split of kFlameScaleJ * Jb for the tensor-core joint regression: [2][16][KB], zero padded
  const int KB = (NB + 15) / 16 * 16;
  fh->KB = KB;
  std::vector<__half> jb16((size_t)2 * 16 * KB, __float2half_rn(0.f));
  for (int i = 0; i < NJ * 3 && i < 16; ++i)
    for (int l = 0; l < NB; ++l) {
      const float sv = Jb[(size_t)i * NB + l] * kFlameScaleJ;
      const __half h = __float2half_rn(sv);
      jb16[(size_t)i * KB + l] = h;
      jb16[(size_t)16 * KB + (size_t)i * KB + l] = __float2half_rn(sv - __half2float(h));
    }
  auto up = [&](float** d, const std::vector<float>& h) -> int {
    MSMD_CHECK_CUDA(cudaMalloc(d, h.size() * sizeof(float)));
    MSMD_CHECK_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    return MSMD_OK;
  };
  int rc = MSMD_OK;
  auto up16 = [&](__half** d, const std::vector<__half>& h) -> int {
    MSMD_CHECK_CUDA(cudaMalloc(d, h.size() * sizeof(__half)));
    MSMD_CHECK_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(__half), cudaMemcpyHostToDevice));
    return MSMD_OK;
  };
  // per-vertex epilogue constants of the tensor-core path, one 32-byte record per vertex (two broadcast LDS.128):
  // w0..w4 | template x y z.  Rows past V are zero (their columns are never stored).
  std::vector<float> vconst((size_t)(fh->N3pad / 3 + 64) * 8, 0.f);
  bool normalised = NJ == 5;
  for (int v = 0; v < V && NJ == 5; ++v) {
    double sum = 0;
    for (int j = 0; j < 5; ++j) { vconst[(size_t)v * 8 + j] = h_w[(size_t)v * 5 + j]; sum += h_w[(size_t)v * 5 + j]; }
    for (int c = 0; c < 3; ++c) vconst[(size_t)v * 8 + 5 + c] = h_t[(size_t)v * 3 + c];
    if (std::fabs(sum - 1.0) > 1e-5) normalised = false;
  }
  fh->weights_normalised = normalised ? 1 : 0;
  if ((rc = up(&fh->basis, basis)) || (rc = up16(&fh->basis_hi, hi)) || (rc = up16(&fh->basis_lo, lo)) ||
      (rc = up(&fh->v_template, h_t)) || (rc = up(&fh->weights, h_w)) || (rc = up(&fh->Jt, Jt)) ||
      (rc = up(&fh->Jb, Jb)) || (rc = up(&fh->vconst, vconst)) || (rc = up16(&fh->Jb16, jb16))) {
    msmd_flame_destroy(fh);
    return rc;
  }
  if (cudaMalloc(&fh->d_parents, 8 * sizeof(int)) != cudaSuccess ||
      cudaMemcpy(fh->d_parents, fh->parents, 8 * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
    msmd_flame_destroy(fh);
    set_error("msmd_flame_create: parents upload failed");
    return MSMD_ERR_CUDA;
  }
  *out = fh;
  return MSMD_OK;
}

extern "C" void msmd_flame_destroy(msmd_flame* fh) {
  if (!fh) return;
  flame_tc_destroy(fh);
  cudaFree(fh->basis); cudaFree(fh->basis_hi); cudaFree(fh->basis_lo); cudaFree(fh->v_template);
  cudaFree(fh->weights); cudaFree(fh->vconst); cudaFree(fh->Jt); cudaFree(fh->Jb); cudaFree(fh->Jb16); cudaFree(fh->d_parents);
  cudaFree(fh->A); cudaFree(fh->A_hi); cudaFree(fh->A_lo); cudaFree(fh->xf);
  delete fh;
}

extern "C" int msmd_flame_decode(msmd_flame* fh, const float* betas, const float* pose, int pose2rot, int64_t B,
                                 float* verts_out, float* joints_out, int impl, void* stream) {
  MSMD_REQUIRE(fh, "msmd_flame_decode: null handle");
  MSMD_REQUIRE(B >= 0, "msmd_flame_decode: negative batch");
  if (B == 0) return MSMD_OK;
  MSMD_REQUIRE(betas && pose && verts_out, "msmd_flame_decode: null tensor pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ensure_workspace(fh, B);
  if (rc) return rc;
  {
    ProfileScope prof("flame_pose", st);
    if (fh->NB % 2 == 0 && fh->Jb16 != nullptr && reinterpret_cast<uintptr_t>(betas) % 8 == 0)   // (float2 loads of the coefficients)
      flame_pose_mma_kernel<5><<<cdiv(B, 32), 256, 0, st>>>(betas, pose, pose2rot, B, fh->NB, fh->KB, fh->Kpad, fh->Jt, fh->Jb16,
                                                           fh->d_parents, fh->A, impl == 0 ? fh->A_hi : nullptr,
                                                           impl == 0 ? fh->A_lo : nullptr, fh->xf, joints_out);
    else
      flame_pose_kernel<5><<<cdiv(B, 8), 256, 0, st>>>(betas, pose, pose2rot, B, fh->NB, fh->Kpad, fh->Jt, fh->Jb,
                                                      fh->d_parents, fh->A, impl == 0 ? fh->A_hi : nullptr,
                                                      impl == 0 ? fh->A_lo : nullptr, fh->xf, joints_out);
    MSMD_CHECK_LAUNCH();
  }
  MSMD_REQUIRE(impl == 0 || impl == 1, "msmd_flame_decode: unknown impl %d", impl);
  if (impl == 0) return flame_decode_tc(fh, B, verts_out, st);
  ProfileScope prof("flame_simt", st);
  dim3 grid(cdiv(fh->N3, FBN), cdiv(B, FBM));
  flame_simt_kernel<5><<<grid, 256, 0, st>>>(fh->A, fh->basis, fh->v_template, fh->weights, fh->xf, B, fh->V,
                                            fh->Kpad, verts_out);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

extern "C" int msmd_vertices2landmarks(const float* verts, const int64_t* faces, const int64_t* lmk_faces_idx,
                                       const float* bary, int64_t B, int V, int L, float* out, void* stream) {
  MSMD_REQUIRE(B >= 0 && L >= 0 && V > 0, "msmd_vertices2landmarks: bad sizes");
  if (B == 0 || L == 0) return MSMD_OK;
  MSMD_REQUIRE(verts && faces && lmk_faces_idx && bary && out, "msmd_vertices2landmarks: null pointer");
  const int64_t n = B * L * 3;
  landmarks_kernel<<<cdiv(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(verts, faces, lmk_faces_idx, bary, B,
                                                                              V, L, out);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

extern "C" int msmd_flame_contour_index(const float* full_pose, int pose2rot, int NJ, const int64_t* neck_chain,
                                        int n_chain, int64_t B, int64_t* out_idx, void* stream) {
  MSMD_REQUIRE(B >= 0 && NJ > 0 && n_chain >= 0, "msmd_flame_contour_index: bad sizes");
  if (B == 0) return MSMD_OK;
  MSMD_REQUIRE(full_pose && neck_chain && out_idx, "msmd_flame_contour_index: null pointer");
  contour_index_kernel<<<cdiv(B, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(full_pose, pose2rot, NJ,
                                                                                  neck_chain, n_chain, B, out_idx);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}
