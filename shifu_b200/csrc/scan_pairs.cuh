// Packed pair scan: the height-scan index chain (isaac_gym.py:393-433) in fp32x2 arithmetic, two envs
// per instruction and one yaw rotation per point pair.  The measured-point grid is symmetric about
// the base (point 186 - pt is -point pt) and round-to-nearest is sign-symmetric, so the rotation of
// the mirror point is EXACTLY the negated rotation of the point: a lane owns a point AND its mirror.
// The per-env scalars travel per env PAIR (e, e+1), so that one 128-bit broadcast load yields two
// packed operands: sA = (2zq_e, 2zq_e1, zq_e, zq_e1), sB = (wq_e, wq_e1, x_e, x_e1), sC = (y_e, y_e1, ..),
// (zq, wq) = normalised yaw quaternion.  The host routes grids that are not point-symmetric to the
// scalar scan.
//
// Used by the fused kernel's scan group (csrc/a1_fused_tma.cuh) and by get_heights_pairs_kernel, the
// fast path of shifu_get_heights (row a5; TerrainGymEnv.get_heights for tasks that keep their own
// Python hooks): the same arithmetic without the rest of the step.  Preconditions of the stand-alone
// kernel (checked by the host, else get_heights_kernel runs): banded scan table, horizontal_scale ==
// 0.1f (3-op constant division), symmetric grid, no cell-index output requested.
#pragma once
#include "a1_kernels.cuh"
#include "f32x2.cuh"

namespace shifu {

// Per-thread packed constants of the index chain.
struct PairScanK {
  f2_t border, rcp, negd, nz, denorm;
  float d;                               // horizontal_scale (exact-division arm)
  int max_px, max_py;                    // clip bounds of the cell index
  unsigned c1;                           // band_w - 1
};

__device__ __forceinline__ PairScanK pair_scan_k(const A1K& k) {
  PairScanK c;
  c.border = pk(k.border, k.border);
  c.rcp = pk(k.hdiv.r, k.hdiv.r);
  c.negd = pk(-k.hdiv.d, -k.hdiv.d);
  c.nz = pk(k.neg_zero, k.neg_zero);
  c.denorm = pk(__int_as_float(1), __int_as_float(1));     // 2^-149
  c.d = k.hdiv.d;
  c.max_px = k.trows - 1;
  c.max_py = k.tcols - 1;
  c.c1 = (unsigned)(k.band_w - 1);
  return c;
}

// Publishes env slot e of a tile (yaw of the PRE-reset pose, base xy) into its pair row of the ring.
template <class CRow>
__device__ __forceinline__ void publish_scan_env(const ScanEnv& ev, int e, float4* sA, float4* sB, CRow* sC) {
  const int q = e >> 1, sl = e & 1;
  float* a = reinterpret_cast<float*>(&sA[q]);
  float* b = reinterpret_cast<float*>(&sB[q]);
  float* c = reinterpret_cast<float*>(&sC[q]);
  a[sl] = ev.z2; a[2 + sl] = ev.z;
  b[sl] = ev.w; b[2 + sl] = ev.x;
  c[sl] = ev.y;
}

// Cell index of a packed pair of positions (ax, ay) [already + base xy + border]: the division by
// horizontal_scale, .long() + clip (isaac_gym.py:416-425) and the banded table offset
// (px>>3)*8*W + py*8 + (px&7)  ==  (px & ~7)*(W-1) + px + 8*py.
template <bool EXACT_DIV>
__device__ __forceinline__ void cell_pair(const PairScanK& c, f2_t ax, f2_t ay, unsigned& i0, unsigned& i1) {
  unsigned px0, px1, py0, py1;
  if (EXACT_DIV) {
    float a0, a1, b0, b1;
    upk(ax, a0, a1); upk(ay, b0, b1);
    // float->uint truncates and saturates at 0
    px0 = min(__float2uint_rz(div_rn(a0, c.d)), (unsigned)c.max_px);
    px1 = min(__float2uint_rz(div_rn(a1, c.d)), (unsigned)c.max_px);
    py0 = min(__float2uint_rz(div_rn(b0, c.d)), (unsigned)c.max_py);
    py1 = min(__float2uint_rz(div_rn(b1, c.d)), (unsigned)c.max_py);
  } else {                         // q0 = x*r; e = fma(-d, q0, x); q = fma(e, r, q0)
    const f2_t qx = mul2(ax, c.rcp), qy = mul2(ay, c.rcp);
    const f2_t fx = fma2(fma2(c.negd, qx, ax), c.rcp, qx), fy = fma2(fma2(c.negd, qy, ay), c.rcp, qy);
    // .long() + clip without the conversion unit: RZ(f * 2^-149) is the denormal whose bit
    // pattern IS trunc(f) for 0 <= f < 2^23 (negative f -> sign bit -> relu -> 0, larger f
    // -> a normal number >= 2^23 -> upper clip); one packed multiply per env pair
    int ix0, ix1, iy0, iy1;
    upk_i(mulrz2(fx, c.denorm), ix0, ix1);
    upk_i(mulrz2(fy, c.denorm), iy0, iy1);
    px0 = (unsigned)__vimin_s32_relu(ix0, c.max_px); px1 = (unsigned)__vimin_s32_relu(ix1, c.max_px);
    py0 = (unsigned)__vimin_s32_relu(iy0, c.max_py); py1 = (unsigned)__vimin_s32_relu(iy1, c.max_py);
  }
  i0 = ((px0 & ~7u) * c.c1 + px0) + (py0 << 3);
  i1 = ((px1 & ~7u) * c.c1 + px1) + (py1 << 3);
}

// Cell indices of scan point (bx, by) [BX, BY, NBY = packed bx, by, -by] and of its mirror point for the
// env pair of ring rows a = sA, b = sB, y = the (y_e, y_e1) half of sC:
// idx = {point e, point e+1, mirror e, mirror e+1}.
template <bool EXACT_DIV>
__device__ __forceinline__ void point_pair_cells(const PairScanK& c, f2_t BX, f2_t BY, f2_t NBY, float4 a, float4 b,
                                                 float2 y, unsigned* idx) {
  const f2_t Z2 = pk(a.x, a.y), Z = pk(a.z, a.w), W = pk(b.x, b.y), X = pk(b.z, b.w), Y = pk(y.x, y.y);
  // quat_apply_yaw (shifu/utils/terrain.py:202-206) on (bx, by, 0):
  //   t = 2(q x b) = (-2z*by, 2z*bx);  out = (b + w*t) + q x t,  q x t = (-z*ty, z*tx)
  // Products that feed an add are written fma(a, b, -0): ptxas contracts
  // mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (single rounding) even under --fmad=false,
  // which flips ~0.3 % of the cell indices; fma(a, b, -0) == RN(a*b) exactly and cannot be
  // contracted again (the -0 comes from a kernel parameter, so it is not constant-folded).
  const f2_t tx = mul2(Z2, NBY), ty = mul2(Z2, BX);
  const f2_t rx = sub2(add2(BX, fma2(W, tx, c.nz)), fma2(Z, ty, c.nz));
  const f2_t ry = add2(add2(BY, fma2(W, ty, c.nz)), fma2(Z, tx, c.nz));
  // + base xy, + border (isaac_gym.py:416-420)
  cell_pair<EXACT_DIV>(c, add2(add2(rx, X), c.border), add2(add2(ry, Y), c.border), idx[0], idx[1]);
  // the mirror point: rotation = (-rx, -ry) exactly, and RN(-r + X) == RN(X - r)
  cell_pair<EXACT_DIV>(c, add2(sub2(X, rx), c.border), add2(sub2(Y, ry), c.border), idx[2], idx[3]);
}

// CTA = 12 warps; tile = 32 envs.  Warp w owns point pairs 32*(w%3).. (a lane = scan point pt and its
// mirror point 186 - pt) for env pairs 4*(w/3) .. +3.
constexpr int SP_THREADS = 384;

__global__ void __launch_bounds__(SP_THREADS, 4)
get_heights_pairs_kernel(const __grid_constant__ A1K k, const float* __restrict__ root, float* __restrict__ mh) {
  // pair rows of the ring (sC without the zb half); double-buffered
  __shared__ float4 sA[2][A1_TILE / 2], sB[2][A1_TILE / 2];
  __shared__ float2 sC[2][A1_TILE / 2];
  const int t = threadIdx.x, sw = t >> 5, lane = t & 31;
  const int raw = 32 * (sw % 3) + lane;
  const bool live = raw <= A1_POINTS / 2;                 // pairs 0..93; 93 is the centre, its own mirror
  const int pt = live ? raw : A1_POINTS / 2;
  const int mir = (A1_POINTS - 1) - 2 * pt;
  const float bx = k.px[pt % A1_NX], by = k.py[pt / A1_NX];
  const f2_t BX = pk(bx, bx), BY = pk(by, by), NBY = pk(-by, -by);
  const PairScanK sk = pair_scan_k(k);
  const short* __restrict__ table = k.table;
  const int tiles = (k.n + A1_TILE - 1) / A1_TILE;

  auto publish = [&](int tile, int buf) {                 // threads 0..31: yaw normalisation of the tile's envs
    if (t < A1_TILE) {
      const int e = tile * A1_TILE + t;
      ScanEnv ev = {0.0f, 0.0f, 1.0f, 0.0f, 0.0f};
      if (e < k.n) ev = make_scan_env(root + ((long long)e * k.root_stride + k.root_offset) * 13);
      publish_scan_env(ev, t, sA[buf], sB[buf], sC[buf]);
    }
  };

  int buf = 0;
  if ((int)blockIdx.x < tiles) publish(blockIdx.x, 0);
  __syncthreads();
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, buf ^= 1) {
    const int next = tile + gridDim.x;
    if (next < tiles) publish(next, buf ^ 1);             // overlaps this tile's arithmetic
    const long long e0 = (long long)tile * A1_TILE;
#pragma unroll
    for (int it = 0; it < 2; ++it) {                      // two items of 2 env pairs x (point, mirror point)
      const int q0 = 4 * (sw / 3) + 2 * it;
      unsigned idx[8];
#pragma unroll
      for (int u = 0; u < 2; ++u)
        point_pair_cells<false>(sk, BX, BY, NBY, sA[buf][q0 + u], sB[buf][q0 + u], sC[buf][q0 + u], idx + 4 * u);
      int h[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) h[u] = __ldg(table + idx[u]);
      if (live) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
#pragma unroll
          for (int m = 0; m < 2; ++m) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const long long e = e0 + 2 * (q0 + u) + r;
              if (e < k.n)
                __stcs(mh + e * A1_POINTS + pt + (m ? mir : 0), mul_rn((float)h[4 * u + 2 * m + r], k.vscale));   // :433
            }
          }
        }
      }
    }
    __syncthreads();                                      // next tile's env pairs are published / this tile's are dead
  }
}

}  // namespace shifu
