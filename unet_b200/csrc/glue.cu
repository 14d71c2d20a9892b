// Memory-bound glue of the decoder, the loss, the optimizers, the layout casts at the API edge and the overlap-tile
// stitching of prediction.  NHWC bf16 activations, 16-byte vector accesses, fp32 math, deterministic reductions.
//
// Replaces: PixelShuffle_ICNR (+ReplicationPad2d+AvgPool2d blur), torch.cat + ReLU of fastai UnetBlock/MergeLayer
// (reference train.py:141 DynamicUnet), CrossEntropyLossFlat(axis=1) fwd+bwd (train.py:195,211), fastai Adam / SGD
// (train.py:218), softmax + numpy sum/count/argmax merge (predict.py:193-203, 284-334).
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "host_util.h"
#include "ptx.cuh"
#include "stream.cuh"

namespace b2u {

static inline int grid_for(long long work_items, int threads, int per_sm = 8) {
  long long b = (work_items + threads - 1) / threads;
  const long long cap = (long long)sm_count() * per_sm;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ------------------------------------------------------------------------------------------------ weight staging
struct WStageItem {
  const float* w;       // fp32 [Cout][Cin][kk]
  const float* bias;    // fp32 [Cout] or null
  const int* row_of_co; // null = identity
  __nv_bfloat16* wf;    // [Cout rows][kk][wf_cinp]
  __nv_bfloat16* wd;    // [Cin][kk][wd_coutp] (flipped taps) or null
  float* bias_rows;     // fp32 [Cout] in GEMM row order, or null
  int Cout, Cin, kk, wf_cinp, wd_coutp;
  float scale;
  int block_start;      // first block of this item in the batched launch
  const float* dscale;  // nullable device scalar on top of `scale` (1/sigma of a spectral-normed weight)
};

// One block = a 32 (output channels) x 32 (input channels) tile of one layer with all kh*kw taps: the fp32 master rows are
// read as contiguous runs, transposed through shared memory and written as 64-byte runs of BOTH bf16 layouts (the
// dgrad layout is the channel transpose of the fprop layout, so a direct scatter would write 2 bytes per sector).
__global__ void __launch_bounds__(256) stage_weights_kernel(const WStageItem* __restrict__ items, int n_items) {
  pdl_enter();
  // binary search for the item owning this block
  int lo = 0, hi = n_items - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (items[mid].block_start <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const WStageItem it = items[lo];
  const float wscale = it.scale * (it.dscale ? __ldg(it.dscale) : 1.f);
  __shared__ __nv_bfloat16 tile[32][32 * 9 + 2];   // +2: odd word stride, conflict-free column reads
  const int kk = it.kk;
  const int tiles_ci = (it.Cin + 31) >> 5;
  const int b = (int)blockIdx.x - it.block_start;
  const int co0 = (b / tiles_ci) * 32, ci0 = (b % tiles_ci) * 32;
  const int nco = min(32, it.Cout - co0), nci = min(32, it.Cin - ci0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int run = nci * kk;
  for (int r = warp; r < nco; r += 8) {
    const float* src = it.w + ((size_t)(co0 + r) * it.Cin + ci0) * kk;
    for (int j = lane; j < run; j += 32) tile[r][j] = __float2bfloat16_rn(src[j] * wscale);
  }
  int row_l = co0 + lane;   // GEMM row of output channel co0 + lane
  if (it.row_of_co && lane < nco) row_l = it.row_of_co[co0 + lane];
  __syncthreads();
  for (int q = warp; q < nco * kk; q += 8) {
    const int r = q / kk, t = q - r * kk;
    const int row = __shfl_sync(0xffffffffu, row_l, r);
    if (lane < nci) it.wf[((size_t)row * kk + t) * it.wf_cinp + ci0 + lane] = tile[r][lane * kk + t];
  }
  if (it.wd) {
    for (int q = warp; q < nci * kk; q += 8) {
      const int ci = q / kk, t = q - ci * kk;
      if (lane < nco) it.wd[((size_t)(ci0 + ci) * kk + (kk - 1 - t)) * it.wd_coutp + row_l] = tile[lane][ci * kk + t];
    }
  }
  if (ci0 == 0 && it.bias && it.bias_rows && warp == 0 && lane < nco) it.bias_rows[row_l] = it.bias[co0 + lane];
}

// ------------------------------------------------------------------------------------------------ decoder glue
// cat[n,Y,X,0:cu]      = blur(PixelShuffle(u))       u: [N,h,w,4cu], channel order (i,j,c)
// cat[n,Y,X,cu:cu+cs]  = act(skip*sscale+sshift)     (sscale null: plain copy)
// cat[n,Y,X,cu+cs:ldc] = 0
// Every thread owns a fixed 8-channel group of the concat, hence a fixed ROLE (shuffle / skip / zero pad): the role
// switch sits outside the pixel loop, the skip constants are loaded once per thread, and the loads of four pixels (up to
// 16 x 16 B for the blurred shuffle) are in flight before the first store.
template <bool kBlur> struct CatRegs { uint4 a, b, d, e; };
template <> struct CatRegs<false> { uint4 a; };

template <bool kBlur>
__global__ void __launch_bounds__(256, 2) shuffle_cat_fwd_kernel(
    const __nv_bfloat16* __restrict__ u, int ldu, int cu, const __nv_bfloat16* __restrict__ skip, int lds,
    int cs, const float* __restrict__ sscale, const float* __restrict__ sshift, int skip_relu,
    __nv_bfloat16* __restrict__ cat, int ldc, int N, int h, int w, int H, int W) {
  pdl_enter();
  // cat is [N, H, W, ldc] with H in {2h, 2h-1}, W in {2w, 2w-1}: an odd skip size crops the last row / column of the
  // upsampled tensor - what fastai's F.interpolate(up_out, skip.shape[-2:], mode='nearest') does for 2h -> 2h-1
  auto ps = [&](int n, int yy, int xx, int c) {
    return ldq(u + ((long long)(n * h + (yy >> 1)) * w + (xx >> 1)) * ldu + (((yy & 1) * 2 + (xx & 1)) * cu + c));
  };
  auto store = [&](int p, int c, const f8& o) { st8(cat + (long long)p * ldc + c, o); };
  struct SkipConsts { f8 sc, sh; };
  // bytes in flight per thread: 4 pixels x 4 loads (blur) or 8 pixels x 1 load
  stream_pixel_groups_xy<kBlur ? 4 : 8, CatRegs<kBlur>>(N, H, W, ldc >> 3,
      [&](int c) {
        // skip role: BatchNorm affine of this thread's channel group (arrays padded to a multiple of 32 floats, b2u.h)
        SkipConsts k;
        if (sscale && c >= cu && c < cu + cs) { k.sc = ldc8(sscale, c - cu, cs); k.sh = ldc8(sshift, c - cu, cs); }
        return k;
      },
      [&](int p, int n, int Y, int X, int c, const SkipConsts&, CatRegs<kBlur>& q) {
        if (c < cu) {
          if constexpr (kBlur) {
            const int y0 = Y > 0 ? Y - 1 : 0, x0 = X > 0 ? X - 1 : 0;
            q.a = ps(n, y0, x0, c); q.b = ps(n, y0, X, c); q.d = ps(n, Y, x0, c); q.e = ps(n, Y, X, c);
          } else {
            q.a = ps(n, Y, X, c);
          }
        } else if (skip && c < cu + cs) {
          q.a = ldq(skip + (long long)p * lds + (c - cu));
        }
      },
      [&](int p, int n, int Y, int X, int c, const SkipConsts& k, const CatRegs<kBlur>& q) {
        f8 o;
        if (c < cu) {
          if constexpr (kBlur) {
            const f8 a = unpack_f8(q.a), b = unpack_f8(q.b), d = unpack_f8(q.d), e = unpack_f8(q.e);
#pragma unroll
            for (int k = 0; k < 8; ++k) o.v[k] = 0.25f * ((a.v[k] + b.v[k]) + (d.v[k] + e.v[k]));
          } else {
            o = unpack_f8(q.a);
          }
        } else if (skip && c < cu + cs) {
          const int sc0 = c - cu;
          o = unpack_f8(q.a);
          if (sscale) {
#pragma unroll
            for (int i = 0; i < 8; ++i) o.v[i] = o.v[i] * k.sc.v[i] + k.sh.v[i];
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (skip_relu) o.v[i] = fmaxf(o.v[i], 0.f);
            if (sc0 + i >= cs) o.v[i] = 0.f;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) o.v[k] = 0.f;
        }
        store(p, c, o);
      });
}

// The blurred variant, blocked 2x2: one thread produces the four concat pixels (2y+a, 2x+b) of one cell (y, x) of the
// pre-shuffle grid for its 8-channel group.  Their 2x2 blur windows overlap - the union is the 3x3 patch of shuffled pixels
// PS[2y-1..2y+1, 2x-1..2x+1] - so a cell costs 9 loads instead of 16 (the per-pixel kernel was bound by load issue, not by
// DRAM).  Same summation order as the per-pixel kernel: bit-identical results.
struct CatBlurRegs { uint4 v[9]; };   // shuffle role: the 3x3 patch, row-major; skip role: v[0..3] = the four skip pixels

__global__ void __launch_bounds__(256, 2) shuffle_cat_blur2x2_kernel(
    const __nv_bfloat16* __restrict__ u, int ldu, int cu, const __nv_bfloat16* __restrict__ skip, int lds,
    int cs, const float* __restrict__ sscale, const float* __restrict__ sshift, int skip_relu,
    __nv_bfloat16* __restrict__ cat, int ldc, int N, int h, int w, int H, int W) {
  pdl_enter();
  auto ps = [&](int n, int yy, int xx, int c) {   // replication pad: row / column -1 is row / column 0
    yy = max(yy, 0); xx = max(xx, 0);
    return ldq(u + ((long long)(n * h + (yy >> 1)) * w + (xx >> 1)) * ldu + (((yy & 1) * 2 + (xx & 1)) * cu + c));
  };
  struct SkipConsts { f8 sc, sh; };
  stream_pixel_groups_xy<1, CatBlurRegs>(N, h, w, ldc >> 3,
      [&](int c) {
        SkipConsts k;
        if (sscale && c >= cu && c < cu + cs) { k.sc = ldc8(sscale, c - cu, cs); k.sh = ldc8(sshift, c - cu, cs); }
        return k;
      },
      [&](int p, int n, int y, int x, int c, const SkipConsts&, CatBlurRegs& q) {
        const int Y = 2 * y, X = 2 * x;
        if (c < cu) {
#pragma unroll
          for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int t = 0; t < 3; ++t) q.v[r * 3 + t] = ps(n, Y - 1 + r, X - 1 + t, c);
        } else if (skip && c < cu + cs) {
#pragma unroll
          for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
              const int yy = min(Y + a, H - 1), xx = min(X + b, W - 1);     // cropped pixels: clamped load, never stored
              q.v[a * 2 + b] = ldq(skip + ((long long)(n * H + yy) * W + xx) * lds + (c - cu));
            }
        }
      },
      [&](int p, int n, int y, int x, int c, const SkipConsts& k, const CatBlurRegs& q) {
        const int Y = 2 * y, X = 2 * x;
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            if (Y + a >= H || X + b >= W) continue;     // odd skip size: last row / column of the upsampled tensor cropped
            f8 o;
            if (c < cu) {
              const f8 pa = unpack_f8(q.v[a * 3 + b]), pb = unpack_f8(q.v[a * 3 + b + 1]);
              const f8 pd = unpack_f8(q.v[(a + 1) * 3 + b]), pe = unpack_f8(q.v[(a + 1) * 3 + b + 1]);
#pragma unroll
              for (int i = 0; i < 8; ++i) o.v[i] = 0.25f * ((pa.v[i] + pb.v[i]) + (pd.v[i] + pe.v[i]));
            } else if (skip && c < cu + cs) {
              const int sc0 = c - cu;
              o = unpack_f8(q.v[a * 2 + b]);
              if (sscale) {
#pragma unroll
                for (int i = 0; i < 8; ++i) o.v[i] = o.v[i] * k.sc.v[i] + k.sh.v[i];
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (skip_relu) o.v[i] = fmaxf(o.v[i], 0.f);
                if (sc0 + i >= cs) o.v[i] = 0.f;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) o.v[i] = 0.f;
            }
            st8(cat + ((long long)(n * H + Y + a) * W + X + b) * ldc + c, o);
          }
      });
}

// du[n,y,x,(i,j,c)] = (u>0) * blur^T(dcat[..., 0:cu])[n, 2y+i, 2x+j, c]
template <bool kBlur> struct ShufBwdRegs { uint4 a, b, d, e, u; };
template <> struct ShufBwdRegs<false> { uint4 a, u; };

// `u` null: the ReLU mask is read from `ucat` (the upsampled tensor itself, same addressing as dcat) - without blur
// cat[n,2y+i,2x+j,c] IS relu(u[n,y,x,(i,j,c)]), so the pre-shuffle activation need not be kept.
template <bool kBlur>
__global__ void __launch_bounds__(256, 2) shuffle_bwd_kernel(
    const __nv_bfloat16* __restrict__ dcat, int ldc, const __nv_bfloat16* __restrict__ u,
    const __nv_bfloat16* __restrict__ ucat, __nv_bfloat16* __restrict__ du, int ldu, int cu, int N, int h, int w,
    int H, int W) {
  pdl_enter();
  // dcat is [N, H, W, ldc] (H in {2h, 2h-1}, W likewise): shuffled pixels beyond it were cropped and get no gradient
  const int gpc = cu >> 3;   // 8-channel groups per (i,j) phase
  auto dc = [&](int n, int yy, int xx, int c) { return ldq(dcat + ((long long)(n * H + yy) * W + xx) * ldc + c); };
  stream_pixel_groups_xy<kBlur ? 3 : 8, ShufBwdRegs<kBlur>>(N, h, w, (4 * cu) >> 3,
      [](int) { return 0; },
      [&](int p, int n, int y, int x, int ch, int, ShufBwdRegs<kBlur>& q) {
        const int ij = (ch >> 3) / gpc, c = ch - ij * cu;
        // out-of-range positions are fetched from a clamped (valid) address and weighted by zero below
        const int Y = min(2 * y + (ij >> 1), H - 1), X = min(2 * x + (ij & 1), W - 1);
        q.u = u ? ldq(u + (long long)p * ldu + ch) : ldq(ucat + ((long long)(n * H + Y) * W + X) * ldc + c);
        q.a = dc(n, Y, X, c);
        if constexpr (kBlur) {
          const int Y1 = min(Y + 1, H - 1), X1 = min(X + 1, W - 1);
          q.b = dc(n, Y, X1, c); q.d = dc(n, Y1, X, c); q.e = dc(n, Y1, X1, c);
        }
      },
      [&](int p, int n, int y, int x, int ch, int, const ShufBwdRegs<kBlur>& q) {
        const int ij = (ch >> 3) / gpc;
        const int Y = 2 * y + (ij >> 1), X = 2 * x + (ij & 1);
        const float inb = (Y < H && X < W) ? 1.f : 0.f;      // cropped shuffled pixel: no gradient
        f8 o = unpack_f8(q.a);
        if constexpr (kBlur) {
          // PS[Y,X] feeds outputs (Y+a, X+b), a,b in {0,1}; the replicated first row/column counts twice
          const float wy0 = ((Y == 0) ? 2.f : 1.f) * inb, wx0 = (X == 0) ? 2.f : 1.f;
          const float hy = (Y + 1 < H) ? inb : 0.f, hx = (X + 1 < W) ? 1.f : 0.f;
          const f8 b = unpack_f8(q.b), d = unpack_f8(q.d), e = unpack_f8(q.e);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float s = wy0 * wx0 * o.v[k];
            s += (wy0 * hx) * b.v[k];
            s += (wx0 * hy) * d.v[k];
            s += (hx * hy) * e.v[k];
            o.v[k] = 0.25f * s;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) o.v[k] *= inb;
        }
        const f8 uv = unpack_f8(q.u);
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = uv.v[k] > 0.f ? o.v[k] : 0.f;
        st8(du + (long long)p * ldu + ch, o);
      });
}

// AvgPool2d(2, ceil_mode=True) on an odd extent averages its last window over the samples that exist; replicating the
// last row / column to an even extent first makes the plain 2x2 mean (four taps x 1/4 folded into the idpath's 1x1
// convolution) produce exactly that: xp[n,y,x] = x[n, min(y,H-1), min(x,W-1)].
__global__ void pad_even_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ xp, int G, int N,
                                    int H, int W, int Hp, int Wp) {
  pdl_enter();
  const long long total = (long long)N * Hp * Wp * G;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i % G);
    long long t = i / G;
    const int xx = (int)(t % Wp); t /= Wp;
    const int yy = (int)(t % Hp);
    const int n = (int)(t / Hp);
    const long long src = (((long long)n * H + min(yy, H - 1)) * W + min(xx, W - 1)) * G + g;
    reinterpret_cast<uint4*>(xp)[i] = __ldg(reinterpret_cast<const uint4*>(x) + src);
  }
}

// its adjoint: every original pixel collects the gradients of its replicas
__global__ void pad_even_bwd_kernel(const __nv_bfloat16* __restrict__ dxp, __nv_bfloat16* __restrict__ dx, int accumulate,
                                    int G, int N, int H, int W, int Hp, int Wp) {
  pdl_enter();
  const long long total = (long long)N * H * W * G;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i % G);
    long long t = i / G;
    const int xx = (int)(t % W); t /= W;
    const int yy = (int)(t % H);
    const int n = (int)(t / H);
    auto at = [&](int y2, int x2) { return ld8(dxp + ((((long long)n * Hp + y2) * Wp + x2) * G + g) * 8); };
    f8 o = at(yy, xx);
    const bool ex = (xx == W - 1) && Wp > W, ey = (yy == H - 1) && Hp > H;
    if (ex) { const f8 a = at(yy, W);
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] += a.v[k]; }
    if (ey) { const f8 a = at(H, xx);
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] += a.v[k]; }
    if (ex && ey) { const f8 a = at(H, W);
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] += a.v[k]; }
    __nv_bfloat16* dst = dx + i * 8;
    if (accumulate) { const f8 old = ld8(dst);
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] += old.v[k]; }
    st8(dst, o);
  }
}

// dst[p, dst_off : dst_off + 8*groups] = src[p, src_off : ...] for every pixel (16-byte groups): MergeLayer(dense=True) of
// the final stage - the image bands are concatenated behind the shuffled channels (fastai unet.py layers.10).
__global__ void copy_lanes_kernel(const __nv_bfloat16* __restrict__ src, int lds, int src_off,
                                  __nv_bfloat16* __restrict__ dst, int ldd, int dst_off, int groups, long long pixels) {
  pdl_enter();
  const long long total = pixels * groups;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < total; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long j = i + k * stride, p = j / groups;
      v[k] = ldq(src + p * lds + src_off + (int)(j - p * groups) * 8);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long j = i + k * stride, p = j / groups;
      *reinterpret_cast<uint4*>(dst + p * ldd + dst_off + (int)(j - p * groups) * 8) = v[k];
    }
  }
  for (; i < total; i += stride) {
    const long long p = i / groups;
    const int g = (int)(i - p * groups);
    *reinterpret_cast<uint4*>(dst + p * ldd + dst_off + g * 8) = ldq(src + p * lds + src_off + g * 8);
  }
}

// ------------------------------------------------------------------------------------------------ small-K pointwise
// out[p, c] = mask(z[p, c]) * sum_{k < K} a[p, k] * w[c][k]     (K <= 8: the input gradient of the 1x1 head, whose GEMM
// K is the number of classes).  Pure streaming: a tensor-core tile would be >99 % padding, so this stays on CUDA cores.
template <int KT>
__global__ void pointwise_smallk_kernel(const __nv_bfloat16* __restrict__ a, int lda, int K,
                                        const __nv_bfloat16* __restrict__ w, int ldw,
                                        const __nv_bfloat16* __restrict__ z, int ldz, __nv_bfloat16* __restrict__ out,
                                        int ldo, int pixels, int C) {
  pdl_enter();
  const int G = ldo >> 3;   // every lane of the output pitch is written (zeros beyond C)
  const int per = (pixels + gridDim.x - 1) / gridDim.x;
  const int p0 = blockIdx.x * per, p1 = min(pixels, p0 + per);
  for (int g0 = 0; g0 < G; g0 += blockDim.x) {
    const int GP = min(G - g0, (int)blockDim.x);
    const int PL = blockDim.x / GP;
    const int pl = threadIdx.x / GP, g = g0 + (threadIdx.x - pl * GP);
    if (pl >= PL) continue;
    const int c = g * 8;
    float wk[KT][8];   // [k][lane]
#pragma unroll
    for (int k = 0; k < KT; ++k)
#pragma unroll
      for (int i = 0; i < 8; ++i)
        wk[k][i] = (k < K && c + i < C) ? __bfloat162float(w[(size_t)(c + i) * ldw + k]) : 0.f;
    auto one = [&](int p, const f8& av, const f8& zv) {
      f8 o;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < KT; ++k) s += av.v[k] * wk[k][i];
        o.v[i] = (!z || zv.v[i] > 0.f) ? s : 0.f;
      }
      st8(out + (long long)p * ldo + c, o);
    };
    int p = p0 + pl;
    for (; p + PL < p1; p += 2 * PL) {   // two pixels in flight per thread
      const f8 a0 = ld8(a + (long long)p * lda), a1 = ld8(a + (long long)(p + PL) * lda);
      f8 z0 = a0, z1 = a1;
      if (z) { z0 = ld8(z + (long long)p * ldz + c); z1 = ld8(z + (long long)(p + PL) * ldz + c); }
      one(p, a0, z0);
      one(p + PL, a1, z1);
    }
    if (p < p1) {
      const f8 a0 = ld8(a + (long long)p * lda);
      f8 z0 = a0;
      if (z) z0 = ld8(z + (long long)p * ldz + c);
      one(p, a0, z0);
    }
  }
}

// ------------------------------------------------------------------------------------------------ layout casts
// raw band value -> the network's input value: the reference reads every GeoTIFF dtype as int32 -> float32
// (data.py:24), divides 16-bit datasets by 255 inside its batch transform (utils.py:248-249, 288-289) and by 255 again
// in fastai's IntToFloatTensor; 8-bit datasets see the second division only.  Two true fp32 divisions, as torch does.
__device__ __forceinline__ float load_raw(const void* __restrict__ x, int dtype, long long i, float div, float div2) {
  float v;
  switch (dtype) {
    case B2U_DT_U8: v = (float)reinterpret_cast<const uint8_t*>(x)[i]; break;
    case B2U_DT_U16: v = (float)reinterpret_cast<const uint16_t*>(x)[i]; break;
    case B2U_DT_I16: v = (float)reinterpret_cast<const int16_t*>(x)[i]; break;
    default: v = reinterpret_cast<const float*>(x)[i]; break;
  }
  return (v / div) / div2;
}

// NCHW (fp32 / uint8 / uint16 / int16, divided by div and div2) -> NHWC bf16 with pitch ld at channel offset ch_off;
// remaining lanes of the 8-channel group(s) touched are zeroed when zero_pad is set.
__global__ void nchw_to_nhwc_kernel(const void* __restrict__ x, int dtype, float div, float div2,
                                    __nv_bfloat16* __restrict__ y, int N, int C, int H, int W, int ld, int ch_off, int Cw) {
  pdl_enter();
  const long long HW = (long long)H * W;
  const long long total = (long long)N * HW;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (long long)gridDim.x * blockDim.x) {
    const long long n = p / HW, hw = p - n * HW;
    __nv_bfloat16* dst = y + p * ld + ch_off;
    for (int c0 = 0; c0 < Cw; c0 += 8) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c0 + k;
        v[k] = 0.f;
        if (c < C) {
          const long long src = (n * C + c) * HW + hw;
          v[k] = load_raw(x, dtype, src, div, div2);
        }
      }
      if (c0 + 8 <= Cw && (((ch_off + c0) & 7) == 0)) {
        uint4 u;
        u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
        u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4*>(dst + c0) = u;
      } else {
        for (int k = 0; k < 8 && c0 + k < Cw; ++k) dst[c0 + k] = __float2bfloat16_rn(v[k]);
      }
    }
  }
}

// im2col of a small-channel NHWC bf16 tensor: y[n, oy, ox, c * ks*ks + ky*ks + kx] = x[n, oy*stride + ky - pad, ox*stride + kx - pad, c]
// (zero outside the image and in the pad lanes up to ldy) - torch.nn.functional.unfold's channel order, which is also the
// order of a conv weight [Cout][Cin][kh][kw] read as [Cout][Cin*kh*kw]: the stem's 3x3 stride-2 convolution over 4 bands
// becomes a 1x1 convolution over 36 "channels" whose rows are whole 32-byte sectors for TMA (the 8-byte pixels of the
// 4-band image were one TMA request each).  A warp owns 32 consecutive output pixels: every lane gathers its pixel's
// taps (one 16-byte load per tap when the input pitch allows) into a row of a shared-memory tile, then the warp copies
// the tile - contiguous in shared AND in global memory - with 16-byte accesses.
__global__ void __launch_bounds__(256) im2col_kernel(const __nv_bfloat16* __restrict__ x, int ldx, int C, int H, int W,
                                                     __nv_bfloat16* __restrict__ y, int ldy, int Ho, int Wo, int ks, int stride,
                                                     int pad, long long total_pix) {
  pdl_enter();
  extern __shared__ __align__(16) unsigned short im2col_sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, KK = ks * ks;
  unsigned short* tile = im2col_sm + (size_t)warp * 32 * ldy;
  unsigned short* row = tile + (size_t)lane * ldy;
  const unsigned short* xs = reinterpret_cast<const unsigned short*>(x);
  const bool vec = (ldx & 7) == 0 && C <= 8;
  const int units = ldy >> 3;
  for (long long base = ((long long)blockIdx.x * 8 + warp) * 32; base < total_pix; base += (long long)gridDim.x * 256) {
    const long long pix = base + lane;
    for (int u = 0; u < units; ++u) reinterpret_cast<uint4*>(row)[u] = make_uint4(0u, 0u, 0u, 0u);
    if (pix < total_pix) {
      const long long n = pix / ((long long)Ho * Wo);
      const int r = (int)(pix - n * Ho * Wo), oy = r / Wo, ox = r - oy * Wo;
      int t = 0;
      for (int ky = 0; ky < ks; ++ky) {
        const int iy = oy * stride + ky - pad;
        for (int kx = 0; kx < ks; ++kx, ++t) {
          const int ix = ox * stride + kx - pad;
          if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
          const unsigned short* src = xs + ((n * H + iy) * W + ix) * ldx;
          if (vec) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(src));
            const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int c = 0; c < 8; ++c)
              if (c < C) row[c * KK + t] = (unsigned short)(w4[c >> 1] >> ((c & 1) * 16));
          } else {
            for (int c = 0; c < C; ++c) row[c * KK + t] = __ldg(src + c);
          }
        }
      }
    }
    __syncwarp();
    const long long left = total_pix - base;
    const int n16 = (int)(left < 32 ? left : 32) * units;
    uint4* dst = reinterpret_cast<uint4*>(y + base * ldy);
    const uint4* srcv = reinterpret_cast<const uint4*>(tile);
    for (int i = lane; i < n16; i += 32) dst[i] = srcv[i];
    __syncwarp();
  }
}

// tile t = raster[:, y0[t]:y0[t]+P, x0[t]:x0[t]+P] / div / div2 -> bf16 NHWC [T,P,P,ld] (crop + input contract + layout cast)
__global__ void crop_tiles_kernel(const void* __restrict__ raster, int dtype, float div, float div2, int C, long long Y, long long X,
                                  const int* __restrict__ ty0, const int* __restrict__ tx0, int T, int P,
                                  __nv_bfloat16* __restrict__ out, int ld) {
  pdl_enter();
  const long long PP = (long long)P * P, total = (long long)T * PP;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i / PP);
    const long long r = i - (long long)t * PP;
    const int yy = (int)(r / P), xx = (int)(r - (long long)yy * P);
    const long long gy = (long long)ty0[t] + yy, gx = (long long)tx0[t] + xx;
    const bool inb = gy >= 0 && gy < Y && gx >= 0 && gx < X;
    __nv_bfloat16* dst = out + i * ld;
    // ld is a multiple of 8 (checked on the host): whole 16-byte stores, zeros in the pad lanes
    for (int c0 = 0; c0 < ld; c0 += 8) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c0 + k;
        v[k] = (c < C && inb) ? load_raw(raster, dtype, ((long long)c * Y + gy) * X + gx, div, div2) : 0.f;
      }
      uint4 u;
      u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
      u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
      *reinterpret_cast<uint4*>(dst + c0) = u;
    }
  }
}

// Source pixel (si, sj) of output pixel (i, j) of a dihedrally transformed P x P tile: bit 2 of `op` flips the last axis
// first, then op & 3 quarter turns of torch.rot90(., k, (-2, -1)).
__device__ __forceinline__ void dihedral_src(int op, int P, int i, int j, int& si, int& sj) {
  int u, v;
  switch (op & 3) {
    case 0: u = i; v = j; break;
    case 1: u = j; v = P - 1 - i; break;
    case 2: u = P - 1 - i; v = P - 1 - j; break;
    default: u = P - 1 - j; v = i; break;
  }
  si = u;
  sj = (op & 4) ? P - 1 - v : v;
}

// One 32 x 32 block of one output plane.  The map is a signed permutation of the two axes, so the source pixels of an
// output block form one axis-aligned 32 x 32 block (hanging over the tile edge when P is not a multiple of 32): it is
// read row by row into shared memory and written back row by row, so that both sides stay coalesced when a quarter
// turn transposes.  Pixels outside the raster read as zero, as in crop_tiles_kernel.
template <typename T>
__device__ __forceinline__ void crop_dihedral_block(const T* __restrict__ src, long long Y, long long X, int y0, int x0,
                                                    int op, int P, int a, int b, T* __restrict__ dst, T* tile) {
  int s0i, s0j, s1i, s1j;
  dihedral_src(op, P, a, b, s0i, s0j);
  dihedral_src(op, P, a + 31, b + 31, s1i, s1j);
  const int ri = min(s0i, s1i), rj = min(s0j, s1j);
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int si = ri + r, sj = rj + (int)threadIdx.x;
    if (si >= 0 && si < P && sj >= 0 && sj < P) {
      const long long gy = (long long)y0 + si, gx = (long long)x0 + sj;
      tile[r * 33 + threadIdx.x] = (gy >= 0 && gy < Y && gx >= 0 && gx < X) ? src[gy * X + gx] : T(0);
    }
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int i = a + r, j = b + (int)threadIdx.x;
    if (i < P && j < P) {
      int si, sj;
      dihedral_src(op, P, i, j, si, sj);
      dst[(long long)i * P + j] = tile[(si - ri) * 33 + (sj - rj)];
    }
  }
}

// grid (tile blocks, C + 1, T): plane c < C of tile t is image band c, plane C its label
template <typename TI, typename TL>
__global__ void __launch_bounds__(256) crop_train_batch_kernel(const TI* __restrict__ raster, const TL* __restrict__ labels,
                                                               int C, long long Y, long long X, const int* __restrict__ ty0,
                                                               const int* __restrict__ tx0, const int* __restrict__ top,
                                                               int P, int nb, TI* __restrict__ x, TL* __restrict__ y) {
  __shared__ __align__(16) unsigned char smem[32 * 33 * 4];
  pdl_enter();
  const int t = blockIdx.z, c = blockIdx.y;
  const int a = (blockIdx.x / nb) * 32, b = (blockIdx.x % nb) * 32;
  const int y0 = ty0[t], x0 = tx0[t], op = top[t];
  const long long PP = (long long)P * P;
  if (c < C)
    crop_dihedral_block(raster + (long long)c * Y * X, Y, X, y0, x0, op, P, a, b, x + ((long long)t * C + c) * PP,
                        reinterpret_cast<TI*>(smem));
  else
    crop_dihedral_block(labels, Y, X, y0, x0, op, P, a, b, y + (long long)t * PP, reinterpret_cast<TL*>(smem));
}

template <typename TI, typename TL>
static cudaError_t launch_crop_train_batch(const void* raster, const void* labels, int C, long long Y, long long X,
                                           const int* y0, const int* x0, const int* op, int T, int P, void* x, void* y,
                                           cudaStream_t st) {
  const int nb = (P + 31) / 32;
  return launch_k(crop_train_batch_kernel<TI, TL>, dim3(nb * nb, C + 1, T), dim3(32, 8), 0, st, (const TI*)raster,
                  (const TL*)labels, C, Y, X, y0, x0, op, P, nb, (TI*)x, (TL*)y);
}

__global__ void nhwc_to_nchw_f32_kernel(const void* __restrict__ x, int is_f32, int ld, float* __restrict__ y, int N,
                                        int C, int H, int W) {
  pdl_enter();
  const long long HW = (long long)H * W;
  const long long total = (long long)N * C * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long hw = i % HW;
    const int c = (int)((i / HW) % C);
    const long long n = i / (HW * C);
    const long long src = (n * HW + hw) * ld + c;
    y[i] = is_f32 ? reinterpret_cast<const float*>(x)[src]
                  : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(x)[src]);
  }
}

// ------------------------------------------------------------------------------------------------ cross entropy
__device__ __forceinline__ float block_sum(float v, float* sh) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sh[w] = v;
  __syncthreads();
  float r = 0.f;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += sh[i];
  __syncthreads();
  return r;  // valid on thread 0
}

__global__ void ce_weight_sum_kernel(const uint8_t* __restrict__ labels, long long P, const float* __restrict__ weight,
                                     int C, float* __restrict__ partial) {
  pdl_enter();
  __shared__ float sh[32];
  float s = 0.f;
  const long long per = (P + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(P, p0 + per);
  for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    const int y = labels[p];
    s += (y < C) ? (weight ? __ldg(weight + y) : 1.f) : 0.f;
  }
  const float r = block_sum(s, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = r;
}

// loss partials + dlogits in one pass. dlogits[p][c] = grad_scale * w[y] * (softmax_c - [c==y]) / wsum
template <int MAXC>
__global__ void ce_fwd_bwd_kernel(const float* __restrict__ logits, int ld, const uint8_t* __restrict__ labels,
                                  long long P, int C, const float* __restrict__ weight,
                                  const float* __restrict__ wsum_partial, int wsum_rows,
                                  __nv_bfloat16* __restrict__ dlogits, int ldg, float* __restrict__ loss_partial,
                                  float grad_scale) {
  pdl_enter();
  __shared__ float sh[32];
  __shared__ float s_wsum;
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < wsum_rows; ++i) t += wsum_partial[i];  // fixed order: every block derives the same value
    s_wsum = t;
  }
  __syncthreads();
  const float inv_wsum = s_wsum > 0.f ? 1.f / s_wsum : 0.f;
  float acc = 0.f;
  const long long per = (P + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(P, p0 + per);
  for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    float z[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? logits[p * ld + c] : -INFINITY;
      m = fmaxf(m, z[c]);
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? __expf(z[c] - m) : 0.f;
      se += z[c];
    }
    const int y = labels[p];
    const bool ok = y < C;
    const float wy = ok ? (weight ? __ldg(weight + y) : 1.f) : 0.f;
    const float inv = 1.f / se;
    if (ok) {
      float py = 0.f;
#pragma unroll
      for (int c = 0; c < MAXC; ++c) py = (c == y) ? z[c] * inv : py;
      acc += -wy * __logf(fmaxf(py, 1e-37f));
    }
    if (dlogits) {
      const float gs = grad_scale * wy * inv_wsum;
      // ldg is a multiple of 8 (checked on the host): 16-byte stores, zeros beyond C
      for (int c0 = 0; c0 < ldg; c0 += 8) {
        float gv[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = c0 + k;
          float zc = 0.f;
#pragma unroll
          for (int q = 0; q < MAXC; ++q) zc = (q == c) ? z[q] : zc;
          gv[k] = (c < C) ? gs * (zc * inv - (c == y ? 1.f : 0.f)) : 0.f;
        }
        uint4 u;
        u.x = pack_bf16x2(gv[0], gv[1]); u.y = pack_bf16x2(gv[2], gv[3]);
        u.z = pack_bf16x2(gv[4], gv[5]); u.w = pack_bf16x2(gv[6], gv[7]);
        *reinterpret_cast<uint4*>(dlogits + p * ldg + c0) = u;
      }
    }
  }
  const float r = block_sum(acc, sh);
  if (threadIdx.x == 0) loss_partial[blockIdx.x] = r;
}

__global__ void ce_finalize_kernel(const float* loss_partial, int rows, const float* wsum_partial, int wsum_rows,
                                   float* loss) {
  pdl_enter();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double l = 0, w = 0;
    for (int i = 0; i < rows; ++i) l += loss_partial[i];
    for (int i = 0; i < wsum_rows; ++i) w += wsum_partial[i];
    loss[0] = w > 0 ? (float)(l / w) : 0.f;
  }
}

// MSELossFlat(axis=1) of the regression variant (train.py:189-192): loss = mean_p (pred_p - target_p)^2 over the
// flattened batch; dpred = grad_scale * 2 (pred - target) / P.  pred is lane 0 of the fp32 head output.
__global__ void mse_fwd_bwd_kernel(const float* __restrict__ pred, int ld, const float* __restrict__ target, long long P,
                                   __nv_bfloat16* __restrict__ dpred, int ldg, float* __restrict__ loss_partial,
                                   float grad_scale) {
  pdl_enter();
  __shared__ float sh[32];
  float acc = 0.f;
  const float gs = grad_scale * 2.f / (float)P;
  const long long per = (P + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(P, p0 + per);
  for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    const float d = pred[p * ld] - target[p];
    acc += d * d;
    if (dpred) {
      uint4 u = make_uint4(pack_bf16x2(gs * d, 0.f), 0u, 0u, 0u);
      for (int c0 = 0; c0 < ldg; c0 += 8) {
        *reinterpret_cast<uint4*>(dpred + p * ldg + c0) = u;
        u.x = 0u;
      }
    }
  }
  const float r = block_sum(acc, sh);
  if (threadIdx.x == 0) loss_partial[blockIdx.x] = r;
}

__global__ void mse_finalize_kernel(const float* loss_partial, int rows, long long P, float* loss) {
  pdl_enter();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double l = 0;
    for (int i = 0; i < rows; ++i) l += loss_partial[i];
    loss[0] = (float)(l / (double)P);
  }
}

// ------------------------------------------------------------------------------------------------ focal / dice losses
// fastai FocalLossFlat(axis=1, gamma, weight=w): per pixel l = w[y] * (-log p_y), pt = exp(-l), f = (1 - pt)^gamma * l.
// Block partials of sum f; b2u_mse_finalize divides by P ('mean') or by 1 ('sum').  dlogits = gs * f'(l) * w[y] *
// (softmax - onehot) with f'(l) = (1 - pt)^gamma * (1 + gamma * pt * l / (1 - pt)).  The second term is the
// gamma * (1-pt)^(gamma-1) * pt * l of the chain rule written so that it stays finite: where 1 - pt == 0 it is 0 (its
// limit for every gamma > 0), so a saturated correct pixel gives 0 and never 0^negative * 0.  Accurate expf / logf: the
// loss is compared with a float64 evaluation at 1e-5.
template <int MAXC>
__global__ void focal_fwd_bwd_kernel(const float* __restrict__ logits, int ld, const uint8_t* __restrict__ labels,
                                     long long P, int C, const float* __restrict__ weight, float gamma,
                                     __nv_bfloat16* __restrict__ dlogits, int ldg, float* __restrict__ loss_partial,
                                     float gs) {
  pdl_enter();
  __shared__ float sh[32];
  float acc = 0.f;
  const long long per = (P + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(P, p0 + per);
  for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    float z[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? logits[p * ld + c] : -INFINITY;
      m = fmaxf(m, z[c]);
    }
    const int y = labels[p];
    const bool ok = y < C;
    float zy = m, se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      zy = (c == y) ? z[c] : zy;
      z[c] = (c < C) ? expf(z[c] - m) : 0.f;
      se += z[c];
    }
    const float wy = ok ? (weight ? __ldg(weight + y) : 1.f) : 0.f;
    const float l = wy * ((m - zy) + logf(se));          // se >= 1: the log is >= 0
    const float omp = -expm1f(-l);                         // 1 - pt
    const float q = powf(omp, gamma);                      // powf(0, 0) = 1: gamma = 0 is plain weighted CE
    acc += q * l;
    if (dlogits) {
      const float dfdl = q * (omp > 0.f ? 1.f + gamma * expf(-l) * (l / omp) : 1.f);
      const float g = gs * dfdl * wy;
      const float inv = 1.f / se;
      for (int c0 = 0; c0 < ldg; c0 += 8) {
        float gv[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = c0 + k;
          float zc = 0.f;
#pragma unroll
          for (int q2 = 0; q2 < MAXC; ++q2) zc = (q2 == c) ? z[q2] : zc;
          gv[k] = (c < C) ? g * (zc * inv - (c == y ? 1.f : 0.f)) : 0.f;
        }
        uint4 u;
        u.x = pack_bf16x2(gv[0], gv[1]); u.y = pack_bf16x2(gv[2], gv[3]);
        u.z = pack_bf16x2(gv[4], gv[5]); u.w = pack_bf16x2(gv[6], gv[7]);
        *reinterpret_cast<uint4*>(dlogits + p * ldg + c0) = u;
      }
    }
  }
  const float r = block_sum(acc, sh);
  if (threadIdx.x == 0) loss_partial[blockIdx.x] = r;
}

// fastai DiceLoss(axis=1, smooth, square_in_union), phase 1.  Grid (bps, N): block (b, n) covers the b-th of bps equal
// pixel ranges of sample n and writes partial[(n*bps + b)*3C + {0, C, 2C} + c] = {sum p_c t_c, sum p_c (or p_c^2),
// sum t_c} over its pixels (t = one-hot label; a label >= C is all zeros).  256 threads; per-thread registers, then
// warp shuffles and the 8 warp sums in warp order: no atomics, the same bits every run.
template <int MAXC>
__global__ void __launch_bounds__(256) dice_stats_kernel(const float* __restrict__ logits, int ld,
                                                         const uint8_t* __restrict__ labels, long long HW, int C,
                                                         int square, float* __restrict__ partial) {
  pdl_enter();
  __shared__ float sh[3 * MAXC][8];
  const int n = blockIdx.y, bps = gridDim.x;
  const long long per = (HW + bps - 1) / bps;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(HW, p0 + per);
  const long long base = (long long)n * HW;
  float si[MAXC], su[MAXC], st[MAXC];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) si[c] = su[c] = st[c] = 0.f;
  for (long long p = base + p0 + threadIdx.x; p < base + p1; p += blockDim.x) {
    float z[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? logits[p * ld + c] : -INFINITY;
      m = fmaxf(m, z[c]);
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? expf(z[c] - m) : 0.f;
      se += z[c];
    }
    const float inv = 1.f / se;
    const int y = labels[p];
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const float pc = z[c] * inv;
      si[c] += (c == y) ? pc : 0.f;
      su[c] += square ? pc * pc : pc;
      st[c] += (c == y) ? 1.f : 0.f;
    }
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    if (c < C) {
      float a = si[c], b = su[c], t = st[c];
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
      }
      if (lane == 0) { sh[c][w] = a; sh[MAXC + c][w] = b; sh[2 * MAXC + c][w] = t; }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) {
    const int k = i / C, c = i - k * C;
    float r = 0.f;
    for (int j = 0; j < 8; ++j) r += sh[k * MAXC + c][j];
    partial[((long long)n * bps + blockIdx.x) * 3 * C + i] = r;
  }
}

// DiceLoss phase 2.  Every block of sample n folds that sample's bps partials in block order (double), so all blocks
// derive the same I_c, U_c = sum p (or p^2) + sum t.  Block 0 of the sample writes loss_partial[n] = sum_c (1 - d_c),
// d_c = (2 I_c + s) / (U_c + s).  With dlogits: g_c = -r (2 t_c (U_c+s) - (2 I_c+s) u'_c) / (U_c+s)^2 (u' = 1, or 2 p_c
// with square_in_union) is pulled back through the softmax: dz_j = p_j (g_j - sum_c p_c g_c).  The grid's x extent
// (blocks per sample of this pass) need not equal bps.
template <int MAXC>
__global__ void __launch_bounds__(256) dice_bwd_kernel(const float* __restrict__ logits, int ld,
                                                       const uint8_t* __restrict__ labels, long long HW, int C,
                                                       int square, const float* __restrict__ partial, int bps,
                                                       float smooth, float r, __nv_bfloat16* __restrict__ dlogits,
                                                       int ldg, float* __restrict__ loss_partial) {
  pdl_enter();
  __shared__ double s_stat[3 * MAXC];
  __shared__ float s_a[MAXC], s_b[MAXC];
  const int n = blockIdx.y;
  if (threadIdx.x < 3 * C) {
    double t = 0.0;
    for (int b = 0; b < bps; ++b) t += partial[((long long)n * bps + b) * 3 * C + threadIdx.x];
    s_stat[threadIdx.x] = t;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    const double den = s_stat[C + c] + s_stat[2 * C + c] + (double)smooth;
    s_a[c] = (float)(2.0 * (double)r / den);
    s_b[c] = (float)((double)r * (2.0 * s_stat[c] + (double)smooth) / (den * den));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double l = 0.0;
    for (int c = 0; c < C; ++c)
      l += 1.0 - (2.0 * s_stat[c] + (double)smooth) / (s_stat[C + c] + s_stat[2 * C + c] + (double)smooth);
    loss_partial[n] = (float)l;
  }
  __syncthreads();
  if (!dlogits) return;
  float a[MAXC], bb[MAXC];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    a[c] = (c < C) ? s_a[c] : 0.f;
    bb[c] = (c < C) ? s_b[c] : 0.f;
  }
  const long long per = (HW + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(HW, p0 + per);
  const long long base = (long long)n * HW;
  for (long long p = base + p0 + threadIdx.x; p < base + p1; p += blockDim.x) {
    float z[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? logits[p * ld + c] : -INFINITY;
      m = fmaxf(m, z[c]);
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] = (c < C) ? expf(z[c] - m) : 0.f;
      se += z[c];
    }
    const float inv = 1.f / se;
    const int y = labels[p];
    float g[MAXC];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      z[c] *= inv;                                                        // p_c (0 beyond C)
      g[c] = bb[c] * (square ? 2.f * z[c] : 1.f) - ((c == y) ? a[c] : 0.f);
      dot += z[c] * g[c];
    }
    for (int c0 = 0; c0 < ldg; c0 += 8) {
      float gv[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c0 + k;
        float pc = 0.f, gc = 0.f;
#pragma unroll
        for (int q = 0; q < MAXC; ++q) {
          pc = (q == c) ? z[q] : pc;
          gc = (q == c) ? g[q] : gc;
        }
        gv[k] = pc * (gc - dot);                                          // 0 beyond C: p_c = 0 there
      }
      uint4 u;
      u.x = pack_bf16x2(gv[0], gv[1]); u.y = pack_bf16x2(gv[2], gv[3]);
      u.z = pack_bf16x2(gv[4], gv[5]); u.w = pack_bf16x2(gv[6], gv[7]);
      *reinterpret_cast<uint4*>(dlogits + p * ldg + c0) = u;
    }
  }
}

// validation sums of the regression metrics (fastai rmse, R2Score; train.py:190): sums[0..3] += {sum (p-t)^2, sum t,
// sum t^2, n} in double.  Block partials are combined by the last block in block order (fixed order: deterministic).
__global__ void regression_sums_kernel(const float* __restrict__ pred, int ld, const float* __restrict__ target,
                                       long long P, double* __restrict__ partial, double* __restrict__ sums,
                                       unsigned int* __restrict__ ticket) {
  pdl_enter();
  __shared__ double sh[3][8];
  __shared__ bool last;
  double a = 0, b = 0, c = 0;
  const long long per = (P + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per, p1 = min(P, p0 + per);
  for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    const double t = target[p], d = (double)pred[p * ld] - t;
    a += d * d; b += t; c += t * t;
  }
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = a; sh[1][w] = b; sh[2][w] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ra = 0, rb = 0, rc = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { ra += sh[0][i]; rb += sh[1][i]; rc += sh[2][i]; }
    partial[blockIdx.x * 3 + 0] = ra; partial[blockIdx.x * 3 + 1] = rb; partial[blockIdx.x * 3 + 2] = rc;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    if (last) {
      __threadfence();
      double s0 = 0, s1 = 0, s2 = 0;
      for (unsigned i = 0; i < gridDim.x; ++i) {
        s0 += __ldcg(partial + i * 3); s1 += __ldcg(partial + i * 3 + 1); s2 += __ldcg(partial + i * 3 + 2);
      }
      sums[0] += s0; sums[1] += s1; sums[2] += s2; sums[3] += (double)P;
      *ticket = 0u;
    }
  }
}

// DiceMulti counts (fastai metrics.py, reached from train.py:196): prediction = argmax_c logits (first maximum wins, as
// torch.argmax); counts[c] += #(pred == c & target == c), counts[C + c] += #(pred == c), counts[2C + c] += #(target == c).
// Integer atomics: the result does not depend on scheduling.
template <int MAXC>
__global__ void dice_counts_kernel(const float* __restrict__ logits, int ld, const uint8_t* __restrict__ labels,
                                   long long P, int C, unsigned long long* __restrict__ counts) {
  pdl_enter();
  __shared__ unsigned int sc[3 * MAXC];
  for (int i = threadIdx.x; i < 3 * MAXC; i += blockDim.x) sc[i] = 0u;
  __syncthreads();
  // a block handles at most 2^31 pixels between flushes: 32-bit shared counters cannot overflow
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long long)gridDim.x * blockDim.x) {
    const float* z = logits + p * ld;
    int best = 0;
    float bv = z[0];
#pragma unroll
    for (int c = 1; c < MAXC; ++c)
      if (c < C) { const float v = z[c]; if (v > bv) { bv = v; best = c; } }
    const int y = labels[p];
    atomicAdd(&sc[MAXC + best], 1u);
    if (y < C) {
      atomicAdd(&sc[2 * MAXC + y], 1u);
      if (y == best) atomicAdd(&sc[y], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * MAXC; i += blockDim.x) {
    const int k = i / MAXC, c = i - k * MAXC;
    if (c < C && sc[i]) atomicAdd(&counts[k * C + c], (unsigned long long)sc[i]);
  }
}

// fp32 <-> bf16 casts of a gradient range (the bf16 copy is what travels over NVLink in the data-parallel all-reduce)
__global__ void cast_f32_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n) {
  pdl_enter();
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    uint2 u;
    u.x = pack_bf16x2(v.x, v.y); u.y = pack_bf16x2(v.z, v.w);
    reinterpret_cast<uint2*>(y)[i] = u;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) y[(n4 << 2) + threadIdx.x] = __float2bfloat16_rn(x[(n4 << 2) + threadIdx.x]);
}
__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, long long n) {
  pdl_enter();
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const uint2 u = reinterpret_cast<const uint2*>(x)[i];
    reinterpret_cast<float4*>(y)[i] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) y[(n4 << 2) + threadIdx.x] = __bfloat162float(x[(n4 << 2) + threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------ optimizers
__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, long long n, float lr, float gs) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] -= lr * gs * g[i];
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, const long long* __restrict__ seg_end,
                            const float* __restrict__ seg_lr, const float* __restrict__ seg_wd, int nseg,
                            const float* __restrict__ hyper) {
  pdl_enter();
  // hyper (device): {mom, sqr_mom, eps, debias1 = 1-mom^step, debias2 = 1-sqr_mom^step, grad_scale}
  const float mom = hyper[0], sqr_mom = hyper[1], eps = hyper[2], debias1 = hyper[3], debias2 = hyper[4], gs = hyper[5];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    int lo = 0, hi = nseg - 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (i < seg_end[mid]) hi = mid; else lo = mid + 1;
    }
    const float lr = seg_lr[lo], wd = seg_wd[lo];
    float pv = p[i];
    const float gv = gs * g[i];
    if (wd != 0.f) pv *= 1.f - lr * wd;
    const float mv = mom * m[i] + (1.f - mom) * gv;
    const float vv = sqr_mom * v[i] + (1.f - sqr_mom) * gv * gv;
    m[i] = mv;
    v[i] = vv;
    pv -= (lr / debias1) * mv / (sqrtf(vv / debias2) + eps);
    p[i] = pv;
  }
}

// ------------------------------------------------------------------------------------------------ stitching
// softmax of tile logits added into the raster accumulators; one launch handles tiles that do not overlap each other.
template <int MAXC>
__global__ void stitch_accumulate_kernel(const float* __restrict__ logits, int ld, int C, int T, int th, int tw,
                                         const int* __restrict__ ty0, const int* __restrict__ tx0,
                                         const int* __restrict__ sel, int n_sel, float* __restrict__ acc,
                                         uint8_t* __restrict__ cnt, long long Y, long long X, long long y_off,
                                         long long x_off, float quant, int raw, const int* __restrict__ n_sel_dev) {
  pdl_enter();
  const long long per_tile = (long long)th * tw;
  // n_sel_dev: the number of selected tiles lives on the device (launches captured in a CUDA graph: the host value
  // n_sel is then only the upper bound the grid was sized for)
  const int nt = sel ? (n_sel_dev ? min(*n_sel_dev, n_sel) : n_sel) : T;
  const long long total = (long long)nt * per_tile;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i / per_tile);
    const int t = sel ? sel[k] : k;
    const long long r = i - (long long)k * per_tile;
    const int yy = (int)(r / tw), xx = (int)(r - (long long)yy * tw);
    const long long gy = (long long)ty0[t] + yy - y_off, gx = (long long)tx0[t] + xx - x_off;
    if (gy < 0 || gy >= Y || gx < 0 || gx >= X) continue;
    const float* z = logits + ((long long)t * per_tile + r) * ld;
    const long long o = gy * X + gx;
    if (raw) {
      // regression merge (predict.py:196-198, 300-302): the network output itself is summed, no softmax
      for (int c = 0; c < C; ++c) acc[(long long)c * Y * X + o] += z[c];
      cnt[o] += 1;
      continue;
    }
    float e[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      e[c] = (c < C) ? z[c] : -INFINITY;
      m = fmaxf(m, e[c]);
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      e[c] = (c < C) ? expf(e[c] - m) : 0.f;
      se += e[c];
    }
    const float inv = 1.f / se;
#pragma unroll
    for (int c = 0; c < MAXC; ++c)
      if (c < C) {
        // quant > 0: the reference's `large_file` mode (predict.py:217-219): prob * 31 -> np.around (half to even) -> int8
        const float pr = e[c] * inv;
        acc[(long long)c * Y * X + o] += quant > 0.f ? rintf(pr * quant) : pr;
      }
    cnt[o] += 1;
  }
}

__global__ void stitch_finalize_kernel(const float* __restrict__ acc, const uint8_t* __restrict__ cnt, int C,
                                       long long YX, uint8_t* __restrict__ mask, int int_div) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < YX; i += (long long)gridDim.x * blockDim.x) {
    const int n = cnt[i];
    int best = 0;
    if (n > 0) {
      // int_div: the int8 sums of `large_file` mode are floor-divided by the count (predict.py:318-323 `//=`)
      float bv = int_div ? floorf(acc[i] / (float)n) : acc[i] / (float)n;
      for (int c = 1; c < C; ++c) {
        float v = acc[(long long)c * YX + i] / (float)n;
        if (int_div) v = floorf(v);
        if (v > bv) { bv = v; best = c; }
      }
    }
    mask[i] = (uint8_t)best;
  }
}

// averaged values of the merge: out[c][i] = acc[c][i] / cnt[i] where tiles were placed, else `nodata` (regression:
// predict.py:307-316 with nodata -9999; averaged class probabilities of `all_classes` / `specific_class`: nodata 0)
__global__ void stitch_finalize_mean_kernel(const float* __restrict__ acc, const uint8_t* __restrict__ cnt, int C,
                                            long long YX, float nodata, float* __restrict__ out) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < YX; i += (long long)gridDim.x * blockDim.x) {
    const int n = cnt[i];
    for (int c = 0; c < C; ++c) out[(long long)c * YX + i] = n > 0 ? acc[(long long)c * YX + i] / (float)n : nodata;
  }
}

// per-tile probabilities (fp32 NCHW) and argmax — what learn.predict hands back per tile
template <int MAXC>
__global__ void softmax_nchw_kernel(const float* __restrict__ logits, int ld, int C, long long tiles, int H, int W,
                                    float* __restrict__ probs, uint8_t* __restrict__ amax) {
  pdl_enter();
  const long long HW = (long long)H * W, total = tiles * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float* z = logits + i * ld;
    float e[MAXC];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      e[c] = (c < C) ? z[c] : -INFINITY;
      m = fmaxf(m, e[c]);
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      e[c] = (c < C) ? expf(e[c] - m) : 0.f;
      se += e[c];
    }
    const float inv = 1.f / se;
    const long long t = i / HW, hw = i - t * HW;
    int best = 0;
    float bv = -1.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      if (c < C) {
        const float pr = e[c] * inv;
        if (probs) probs[(t * C + c) * HW + hw] = pr;
        if (pr > bv) { bv = pr; best = c; }
      }
    }
    if (amax) amax[i] = (uint8_t)best;
  }
}

// Confusion counts of a predicted class map against a truth class map (sklearn.metrics.confusion_matrix orientation:
// bin truth * C + pred).  Block (x, t) owns rows [x * rows, (x + 1) * rows) of image t and a warp one row at a time, so
// a block's joint counts are also the histograms of its image.  Land-cover maps put almost every pixel into two or
// three bins, which serialises per-pixel shared-memory atomics; so the counts of a block are privatised twice:
//   C <= 4 (<= 16 bins): in registers, as 8-bit fields of two 64-bit words (one shift and one add per pixel), spilled
//     to 32-bit register totals every <= 255 pixels and reduced over the warp with redux.sync at the end;
//   C > 4: warp-aggregated shared-memory increments, one atomic per distinct bin of a warp (__match_any_sync + __popc).
// Integer counts throughout: the result is the same bits for any grid and any schedule.
struct RegBins {
  unsigned long long lo = 0, hi = 0;   // bins 0..7 and 8..15, one byte each
  unsigned tot[16] = {};
  unsigned skip = 0;
  int pend = 0;                        // pixels in the byte fields since the last spill (<= 255)
  __device__ __forceinline__ void px(unsigned t, unsigned p, unsigned C) {
    if (t < C && p < C) {
      const unsigned b = t * C + p;
      const unsigned long long s = 1ull << ((b & 7) << 3);
      lo += b < 8 ? s : 0ull;
      hi += b < 8 ? 0ull : s;
    } else {
      ++skip;
    }
  }
  __device__ __forceinline__ void spill() {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      tot[k] += (unsigned)(lo >> (8 * k)) & 255u;
      tot[8 + k] += (unsigned)(hi >> (8 * k)) & 255u;
    }
    lo = hi = 0;
    pend = 0;
  }
  __device__ __forceinline__ void done(int n) {
    pend += n;
    if (pend > 255 - 16) spill();
  }
};

struct SharedBins {
  unsigned* bins;
  unsigned skip = 0;
  __device__ __forceinline__ void px(unsigned t, unsigned p, unsigned C) {
    const unsigned key = (t < C && p < C) ? t * C + p : 0xffffu;
    const unsigned peers = __match_any_sync(__activemask(), key);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) {
      if (key != 0xffffu) atomicAdd(&bins[key], (unsigned)__popc(peers));
      else skip += __popc(peers);
    }
  }
  __device__ __forceinline__ void done(int) {}
};

template <class Bins>
__device__ __forceinline__ void bins_add16(Bins& c, uint4 t, uint4 p, unsigned C) {
  const unsigned tw[4] = {t.x, t.y, t.z, t.w}, pw[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
  for (int w = 0; w < 4; ++w)
#pragma unroll
    for (int k = 0; k < 4; ++k) c.px((tw[w] >> (8 * k)) & 255u, (pw[w] >> (8 * k)) & 255u, C);
  c.done(16);
}

template <bool SMALL>
__global__ void __launch_bounds__(256) confusion_counts_kernel(const uint8_t* __restrict__ pred, long long pp, long long ps,
                                                               const uint8_t* __restrict__ truth, long long tp, long long ts,
                                                               int H, int W, int C, int rows,
                                                               unsigned long long* __restrict__ joint,
                                                               unsigned* __restrict__ tile_hist,
                                                               unsigned long long* __restrict__ skipped) {
  __shared__ unsigned sj[32 * 32];
  __shared__ unsigned sskip;
  pdl_enter();
  const int NB = C * C;
  for (int i = threadIdx.x; i < NB; i += blockDim.x) sj[i] = 0u;
  if (threadIdx.x == 0) sskip = 0u;
  __syncthreads();
  typename std::conditional<SMALL, RegBins, SharedBins>::type c;
  if constexpr (!SMALL) c.bins = sj;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int t = blockIdx.y;
  const int y1 = min(H, (blockIdx.x + 1) * rows);
  for (int y = blockIdx.x * rows + warp; y < y1; y += nw) {
    const uint8_t* p = pred + t * ps + y * pp;
    const uint8_t* q = truth + t * ts + y * tp;
    // 16-byte loads from the first 16-byte boundary of the row when both rows sit at the same offset from it
    int head = (int)((16 - (reinterpret_cast<uintptr_t>(p) & 15)) & 15);
    if ((reinterpret_cast<uintptr_t>(p) ^ reinterpret_cast<uintptr_t>(q)) & 15) head = W;
    head = min(head, W);
    const int nv = (W - head) >> 4;
    for (int x = lane; x < head; x += 32) { c.px(__ldg(q + x), __ldg(p + x), C); c.done(1); }
    const uint4* pv = reinterpret_cast<const uint4*>(p + head);
    const uint4* qv = reinterpret_cast<const uint4*>(q + head);
    int v = lane;
    for (; v + 96 < nv; v += 128) {     // four chunk pairs in flight per lane
      uint4 a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { a[u] = __ldg(qv + v + 32 * u); b[u] = __ldg(pv + v + 32 * u); }
#pragma unroll
      for (int u = 0; u < 4; ++u) bins_add16(c, a[u], b[u], C);
    }
    for (; v < nv; v += 32) bins_add16(c, __ldg(qv + v), __ldg(pv + v), C);
    for (int x = head + 16 * nv + lane; x < W; x += 32) { c.px(__ldg(q + x), __ldg(p + x), C); c.done(1); }
  }
  if constexpr (SMALL) {
    c.spill();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const unsigned s = __reduce_add_sync(0xffffffffu, c.tot[k]);
      if (lane == 0 && k < NB && s) atomicAdd(&sj[k], s);
    }
  }
  const unsigned sk = __reduce_add_sync(0xffffffffu, c.skip);
  if (lane == 0 && sk) atomicAdd(&sskip, sk);
  __syncthreads();
  for (int i = threadIdx.x; i < NB; i += blockDim.x)
    if (sj[i]) atomicAdd(&joint[i], (unsigned long long)sj[i]);
  if (tile_hist) {
    // [t][0][c]: truth histogram (row sums), [t][1][c]: prediction histogram (column sums)
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
      const int k = i / C, cl = i - k * C;
      unsigned s = 0;
      for (int j = 0; j < C; ++j) s += k == 0 ? sj[cl * C + j] : sj[j * C + cl];
      if (s) atomicAdd(&tile_hist[((long long)t * 2 + k) * C + cl], s);
    }
  }
  if (threadIdx.x == 0 && sskip) atomicAdd(skipped, (unsigned long long)sskip);
}

}  // namespace b2u

using namespace b2u;
typedef const __nv_bfloat16* cbf;
typedef __nv_bfloat16* bf;

extern "C" int b2u_stage_weights(const b2u_wstage_item* items_dev, int32_t n_items, int32_t total_blocks,
                                 void* stream) {
  B2U_CHECK_ARG(items_dev && n_items > 0 && total_blocks > 0, "stage_weights: bad argument");
  static_assert(sizeof(b2u_wstage_item) == sizeof(WStageItem), "b2u_wstage_item layout drifted");
  launch_k(stage_weights_kernel, dim3(total_blocks), dim3(256), 0, (cudaStream_t)stream, reinterpret_cast<const WStageItem*>(items_dev),
                                                                      n_items);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_shuffle_cat_fwd_crop(const void* u, int32_t ldu, int32_t cu, int32_t blur, const void* skip,
                                        int32_t lds, int32_t cs, const float* sscale, const float* sshift,
                                        int32_t skip_relu, void* cat, int32_t ldc, int32_t N, int32_t h, int32_t w,
                                        int32_t Ho, int32_t Wo, void* stream) {
  B2U_CHECK_ARG(u && cat && cu > 0 && cu % 8 == 0 && ldu % 8 == 0 && ldc % 8 == 0 && 4 * cu <= ldu && cu <= ldc,
                "shuffle_cat_fwd: bad argument");
  B2U_CHECK_ARG(!skip || (lds % 8 == 0 && cs > 0 && cu + cs <= ldc), "shuffle_cat_fwd: bad skip");
  B2U_CHECK_ARG(!sscale || sshift, "shuffle_cat_fwd: sscale without sshift");
  B2U_CHECK_ARG((Ho == 2 * h || Ho == 2 * h - 1) && (Wo == 2 * w || Wo == 2 * w - 1) && Ho > 0 && Wo > 0,
                "shuffle_cat_fwd: output %dx%d is neither the upsampled size %dx%d nor one less", Ho, Wo, 2 * h, 2 * w);
  const long long items = (long long)N * Ho * Wo * (ldc / 8);
  // 2 resident blocks per SM (register budget of the 4- or 8-pixel load batches): one block per slot, one range each
  const dim3 grid(grid_for(items, 256, 2));
  static const bool per_pixel = getenv("B2U_SHUFFLE_PER_PIXEL") != nullptr;   // A/B switch
  if (blur && !per_pixel)
    launch_k(shuffle_cat_blur2x2_kernel, dim3(grid_for((long long)N * h * w * (ldc / 8), 256, 2)), dim3(256), 0,
             (cudaStream_t)stream, (cbf)u, ldu, cu, (cbf)skip, lds, cs, sscale, sshift, skip_relu, (bf)cat, ldc, N, h, w, Ho,
             Wo);
  else if (blur)
    launch_k(shuffle_cat_fwd_kernel<true>, grid, dim3(256), 0, (cudaStream_t)stream, (cbf)u, ldu, cu, (cbf)skip, lds, cs,
             sscale, sshift, skip_relu, (bf)cat, ldc, N, h, w, Ho, Wo);
  else
    launch_k(shuffle_cat_fwd_kernel<false>, grid, dim3(256), 0, (cudaStream_t)stream, (cbf)u, ldu, cu, (cbf)skip, lds, cs,
             sscale, sshift, skip_relu, (bf)cat, ldc, N, h, w, Ho, Wo);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_shuffle_cat_fwd(const void* u, int32_t ldu, int32_t cu, int32_t blur, const void* skip, int32_t lds,
                                   int32_t cs, const float* sscale, const float* sshift, int32_t skip_relu, void* cat,
                                   int32_t ldc, int32_t N, int32_t h, int32_t w, void* stream) {
  return b2u_shuffle_cat_fwd_crop(u, ldu, cu, blur, skip, lds, cs, sscale, sshift, skip_relu, cat, ldc, N, h, w, 2 * h,
                                  2 * w, stream);
}

static int shuffle_bwd_impl(const void* dcat, int32_t ldc, const void* u, const void* ucat, void* du, int32_t ldu,
                            int32_t cu, int32_t blur, int32_t N, int32_t h, int32_t w, int32_t Ho, int32_t Wo,
                            void* stream) {
  B2U_CHECK_ARG((Ho == 2 * h || Ho == 2 * h - 1) && (Wo == 2 * w || Wo == 2 * w - 1) && Ho > 0 && Wo > 0,
                "shuffle_bwd: gradient size %dx%d is neither the upsampled size %dx%d nor one less", Ho, Wo, 2 * h, 2 * w);
  B2U_CHECK_ARG(dcat && (u || ucat) && du && cu % 8 == 0 && ldu % 8 == 0 && ldc % 8 == 0, "shuffle_bwd: bad argument");
  B2U_CHECK_ARG(u || !blur, "shuffle_bwd: the mask can only come from the upsampled tensor when there is no blur");
  const long long items = (long long)N * h * w * (4 * cu / 8);
  const dim3 grid(grid_for(items, 256, 2));
  if (blur)
    launch_k(shuffle_bwd_kernel<true>, grid, dim3(256), 0, (cudaStream_t)stream, (cbf)dcat, ldc, (cbf)u, (cbf)ucat, (bf)du,
             ldu, cu, N, h, w, Ho, Wo);
  else
    launch_k(shuffle_bwd_kernel<false>, grid, dim3(256), 0, (cudaStream_t)stream, (cbf)dcat, ldc, (cbf)u, (cbf)ucat, (bf)du,
             ldu, cu, N, h, w, Ho, Wo);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_shuffle_bwd(const void* dcat, int32_t ldc, const void* u, void* du, int32_t ldu, int32_t cu,
                               int32_t blur, int32_t N, int32_t h, int32_t w, void* stream) {
  B2U_CHECK_ARG(u != nullptr, "shuffle_bwd: null u");
  return shuffle_bwd_impl(dcat, ldc, u, nullptr, du, ldu, cu, blur, N, h, w, 2 * h, 2 * w, stream);
}

extern "C" int b2u_shuffle_bwd_crop(const void* dcat, int32_t ldc, const void* u, void* du, int32_t ldu, int32_t cu,
                                    int32_t blur, int32_t N, int32_t h, int32_t w, int32_t Ho, int32_t Wo,
                                    void* stream) {
  B2U_CHECK_ARG(u != nullptr, "shuffle_bwd: null u");
  return shuffle_bwd_impl(dcat, ldc, u, nullptr, du, ldu, cu, blur, N, h, w, Ho, Wo, stream);
}

extern "C" int b2u_shuffle_bwd_from_cat(const void* dcat, const void* cat, int32_t ldc, void* du, int32_t ldu, int32_t cu,
                                        int32_t N, int32_t h, int32_t w, void* stream) {
  B2U_CHECK_ARG(cat != nullptr, "shuffle_bwd_from_cat: null cat");
  return shuffle_bwd_impl(dcat, ldc, nullptr, cat, du, ldu, cu, 0, N, h, w, 2 * h, 2 * w, stream);
}

extern "C" int b2u_pad_even_fwd(const void* x, void* xp, int32_t ld, int32_t N, int32_t H, int32_t W, void* stream) {
  B2U_CHECK_ARG(x && xp && ld % 8 == 0 && N > 0 && H > 0 && W > 0, "pad_even_fwd: bad argument");
  const int Hp = H + (H & 1), Wp = W + (W & 1);
  const long long items = (long long)N * Hp * Wp * (ld / 8);
  launch_k(pad_even_fwd_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, (cbf)x, (bf)xp, ld / 8, N, H,
           W, Hp, Wp);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_pad_even_bwd(const void* dxp, void* dx, int32_t accumulate, int32_t ld, int32_t N, int32_t H,
                                int32_t W, void* stream) {
  B2U_CHECK_ARG(dxp && dx && ld % 8 == 0 && N > 0 && H > 0 && W > 0, "pad_even_bwd: bad argument");
  const int Hp = H + (H & 1), Wp = W + (W & 1);
  const long long items = (long long)N * H * W * (ld / 8);
  launch_k(pad_even_bwd_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, (cbf)dxp, (bf)dx,
           accumulate, ld / 8, N, H, W, Hp, Wp);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_copy_lanes(const void* src, int32_t lds, int32_t src_off, void* dst, int32_t ldd, int32_t dst_off,
                              int32_t lanes, int64_t pixels, void* stream) {
  B2U_CHECK_ARG(src && dst && lanes > 0 && lanes % 8 == 0 && lds % 8 == 0 && ldd % 8 == 0 && src_off % 8 == 0 &&
                dst_off % 8 == 0 && src_off + lanes <= lds && dst_off + lanes <= ldd, "copy_lanes: bad argument");
  const long long items = pixels * (lanes / 8);
  launch_k(copy_lanes_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, (cbf)src, lds, src_off,
           (bf)dst, ldd, dst_off, lanes / 8, (long long)pixels);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_pointwise_smallk(const void* a, int32_t lda, int32_t K, const void* w, int32_t ldw, const void* z,
                                    int32_t ldz, void* out, int32_t ldo, int64_t pixels, int32_t C, void* stream) {
  B2U_CHECK_ARG(a && w && out && K >= 1 && K <= 8 && lda >= 8 && lda % 8 == 0 && ldo % 8 == 0 && C <= ldo &&
                    (!z || ldz % 8 == 0) && pixels < (1ll << 31),
                "pointwise_smallk: bad argument (K must be <= 8)");
  const long long items = pixels * (ldo / 8);
  const int grid = grid_for(items, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (K <= 2)
    launch_k(pointwise_smallk_kernel<2>, dim3(grid), dim3(256), 0, st, (cbf)a, lda, K, (cbf)w, ldw, (cbf)z, ldz, (bf)out, ldo, (int)pixels, C);
  else if (K <= 4)
    launch_k(pointwise_smallk_kernel<4>, dim3(grid), dim3(256), 0, st, (cbf)a, lda, K, (cbf)w, ldw, (cbf)z, ldz, (bf)out, ldo, (int)pixels, C);
  else
    launch_k(pointwise_smallk_kernel<8>, dim3(grid), dim3(256), 0, st, (cbf)a, lda, K, (cbf)w, ldw, (cbf)z, ldz, (bf)out, ldo, (int)pixels, C);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_nchw_to_nhwc(const void* x, int32_t x_dtype, float div, float div2, void* y, int32_t N, int32_t C,
                                int32_t H, int32_t W, int32_t ld, int32_t ch_off, int32_t write_c, void* stream) {
  B2U_CHECK_ARG(x && y && C > 0 && write_c >= C && ch_off + write_c <= ld, "nchw_to_nhwc: bad argument");
  B2U_CHECK_ARG(x_dtype >= B2U_DT_F32 && x_dtype <= B2U_DT_I16 && div != 0.f && div2 != 0.f,
                "nchw_to_nhwc: x_dtype=%d (0 f32, 1 u8, 2 u16, 3 i16) / divisors invalid", x_dtype);
  const long long items = (long long)N * H * W;
  launch_k(nchw_to_nhwc_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, x, x_dtype, div, div2, (bf)y, N, C, H, W,
           ld, ch_off, write_c);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_im2col(const void* x, int32_t ldx, int32_t C, int32_t N, int32_t H, int32_t W, int32_t ks, int32_t stride,
                          int32_t pad, void* y, int32_t ldy, void* stream) {
  B2U_CHECK_ARG(x && y && C > 0 && C <= ldx && N > 0 && H > 0 && W > 0 && ks >= 1 && stride >= 1 && pad >= 0, "im2col: bad argument");
  B2U_CHECK_ARG(ldy % 8 == 0 && ldy >= C * ks * ks, "im2col: ldy=%d must be a multiple of 8 and hold C*ks*ks=%d lanes", ldy, C * ks * ks);
  const int Ho = (H + 2 * pad - ks) / stride + 1, Wo = (W + 2 * pad - ks) / stride + 1;
  B2U_CHECK_ARG(Ho > 0 && Wo > 0, "im2col: empty output");
  const long long pixels = (long long)N * Ho * Wo;
  const size_t smem = (size_t)256 * ldy * 2;
  B2U_CHECK_ARG(smem <= 48 * 1024, "im2col: ldy=%d too wide for the shared-memory tile", ldy);
  launch_k(im2col_kernel, dim3(grid_for(pixels, 256)), dim3(256), smem, (cudaStream_t)stream, (const __nv_bfloat16*)x, ldx, C, H, W,
           (bf)y, ldy, Ho, Wo, ks, stride, pad, pixels);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_crop_tiles(const void* raster, int32_t r_dtype, float div, float div2, int32_t C, int64_t Y, int64_t X,
                              const int32_t* y0, const int32_t* x0, int32_t T, int32_t P, void* out, int32_t ld,
                              void* stream) {
  B2U_CHECK_ARG(raster && y0 && x0 && out && C > 0 && C <= ld && ld % 8 == 0 && T > 0 && P > 0, "crop_tiles: bad argument");
  B2U_CHECK_ARG(r_dtype >= B2U_DT_F32 && r_dtype <= B2U_DT_I16 && div != 0.f && div2 != 0.f,
                "crop_tiles: r_dtype=%d (0 f32, 1 u8, 2 u16, 3 i16) / divisors invalid", r_dtype);
  const long long items = (long long)T * P * P;
  launch_k(crop_tiles_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, raster, r_dtype, div, div2, C, Y, X, y0,
           x0, T, P, (bf)out, ld);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_crop_train_batch(const void* raster, int32_t r_dtype, int32_t C, int64_t Y, int64_t X, const void* labels,
                                    int32_t l_dtype, const int32_t* y0, const int32_t* x0, const int32_t* op, int32_t T,
                                    int32_t P, void* x, void* y, void* stream) {
  B2U_CHECK_ARG(raster && labels && y0 && x0 && op && x && y, "crop_train_batch: null argument");
  B2U_CHECK_ARG(C > 0 && C < 65535 && T > 0 && T <= 65535 && P > 0 && P <= Y && P <= X && (long long)P * P < (1ll << 31),
                "crop_train_batch: C=%d T=%d P=%d Y=%lld X=%lld out of range", C, T, P, (long long)Y, (long long)X);
  B2U_CHECK_ARG(r_dtype >= B2U_DT_U8 && r_dtype <= B2U_DT_I16,
                "crop_train_batch: r_dtype=%d (1 u8, 2 u16, 3 i16)", r_dtype);
  B2U_CHECK_ARG(l_dtype == B2U_DT_U8 || l_dtype == B2U_DT_F32, "crop_train_batch: l_dtype=%d (0 f32, 1 u8)", l_dtype);
  const cudaStream_t st = (cudaStream_t)stream;
  const bool f = l_dtype == B2U_DT_F32;
  switch (r_dtype) {
    case B2U_DT_U8:
      f ? launch_crop_train_batch<uint8_t, float>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st)
        : launch_crop_train_batch<uint8_t, uint8_t>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st);
      break;
    case B2U_DT_U16:
      f ? launch_crop_train_batch<uint16_t, float>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st)
        : launch_crop_train_batch<uint16_t, uint8_t>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st);
      break;
    default:
      f ? launch_crop_train_batch<int16_t, float>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st)
        : launch_crop_train_batch<int16_t, uint8_t>(raster, labels, C, Y, X, y0, x0, op, T, P, x, y, st);
  }
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_nhwc_to_nchw_f32(const void* x, int32_t x_is_f32, int32_t ld, float* y, int32_t N, int32_t C,
                                    int32_t H, int32_t W, void* stream) {
  B2U_CHECK_ARG(x && y && C > 0 && C <= ld, "nhwc_to_nchw_f32: bad argument");
  const long long items = (long long)N * C * H * W;
  launch_k(nhwc_to_nchw_f32_kernel, dim3(grid_for(items, 256)), dim3(256), 0, (cudaStream_t)stream, x, x_is_f32, ld, y, N, C, H, W);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_ce_weight_sum(const uint8_t* labels, int64_t P, const float* weight, int32_t C, float* wsum_partial,
                                 int32_t rows, void* stream) {
  B2U_CHECK_ARG(labels && wsum_partial && rows > 0 && C > 0, "ce_weight_sum: bad argument");
  launch_k(ce_weight_sum_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, labels, P, weight, C, wsum_partial);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_ce_fwd_bwd(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C,
                              const float* weight, const float* wsum_partial, int32_t wsum_rows, void* dlogits,
                              int32_t ldg, float* loss_partial, int32_t rows, float grad_scale, void* stream) {
  B2U_CHECK_ARG(logits && labels && wsum_partial && loss_partial && rows > 0, "ce_fwd_bwd: bad argument");
  B2U_CHECK_ARG(C >= 1 && C <= 32 && C <= ld && (!dlogits || (ldg >= C && ldg % 8 == 0)),
                "ce_fwd_bwd: C=%d ld=%d ldg=%d unsupported (ldg must be a multiple of 8)", C, ld, ldg);
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 8)
    launch_k(ce_fwd_bwd_kernel<8>, dim3(rows), dim3(256), 0, st, logits, ld, labels, P, C, weight, wsum_partial, wsum_rows, (bf)dlogits,
                                               ldg, loss_partial, grad_scale);
  else
    launch_k(ce_fwd_bwd_kernel<32>, dim3(rows), dim3(256), 0, st, logits, ld, labels, P, C, weight, wsum_partial, wsum_rows, (bf)dlogits,
                                                ldg, loss_partial, grad_scale);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_ce_finalize(const float* loss_partial, int32_t rows, const float* wsum_partial, int32_t wsum_rows,
                               float* loss, void* stream) {
  B2U_CHECK_ARG(loss_partial && wsum_partial && loss, "ce_finalize: bad argument");
  launch_k(ce_finalize_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, loss_partial, rows, wsum_partial, wsum_rows, loss);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_mse_fwd_bwd(const float* pred, int32_t ld, const float* target, int64_t P, void* dpred, int32_t ldg,
                               float* loss_partial, int32_t rows, float grad_scale, void* stream) {
  B2U_CHECK_ARG(pred && target && loss_partial && rows > 0 && P > 0 && ld >= 1, "mse_fwd_bwd: bad argument");
  B2U_CHECK_ARG(!dpred || (ldg >= 8 && ldg % 8 == 0), "mse_fwd_bwd: ldg=%d must be a positive multiple of 8", ldg);
  launch_k(mse_fwd_bwd_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, pred, ld, target, (long long)P, (bf)dpred, ldg,
           loss_partial, grad_scale);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_mse_finalize(const float* loss_partial, int32_t rows, int64_t P, float* loss, void* stream) {
  B2U_CHECK_ARG(loss_partial && loss && rows > 0 && P > 0, "mse_finalize: bad argument");
  launch_k(mse_finalize_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, loss_partial, rows, (long long)P, loss);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_focal_fwd_bwd(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C,
                                 const float* weight, float gamma, int32_t mean, void* dlogits, int32_t ldg,
                                 float* loss_partial, int32_t rows, float grad_scale, void* stream) {
  B2U_CHECK_ARG(logits && labels && loss_partial && rows > 0 && P > 0 && gamma >= 0.f, "focal_fwd_bwd: bad argument");
  B2U_CHECK_ARG(C >= 1 && C <= 32 && C <= ld && (!dlogits || (ldg >= C && ldg % 8 == 0)),
                "focal_fwd_bwd: C=%d ld=%d ldg=%d unsupported (ldg must be a multiple of 8)", C, ld, ldg);
  cudaStream_t st = (cudaStream_t)stream;
  const float gs = mean ? (float)((double)grad_scale / (double)P) : grad_scale;
  if (C <= 8)
    launch_k(focal_fwd_bwd_kernel<8>, dim3(rows), dim3(256), 0, st, logits, ld, labels, (long long)P, C, weight, gamma,
             (bf)dlogits, ldg, loss_partial, gs);
  else
    launch_k(focal_fwd_bwd_kernel<32>, dim3(rows), dim3(256), 0, st, logits, ld, labels, (long long)P, C, weight, gamma,
             (bf)dlogits, ldg, loss_partial, gs);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_dice_stats(const float* logits, int32_t ld, const uint8_t* labels, int32_t N, int64_t HW, int32_t C,
                              int32_t square_in_union, float* partial, int32_t blocks_per_sample, void* stream) {
  B2U_CHECK_ARG(logits && labels && partial && N > 0 && N <= 65535 && HW > 0 && blocks_per_sample > 0,
                "dice_stats: bad argument");
  B2U_CHECK_ARG(C >= 1 && C <= 32 && C <= ld, "dice_stats: C=%d ld=%d unsupported", C, ld);
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid(blocks_per_sample, N);
  if (C <= 8)
    launch_k(dice_stats_kernel<8>, grid, dim3(256), 0, st, logits, ld, labels, (long long)HW, C, square_in_union, partial);
  else
    launch_k(dice_stats_kernel<32>, grid, dim3(256), 0, st, logits, ld, labels, (long long)HW, C, square_in_union, partial);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_dice_bwd(const float* logits, int32_t ld, const uint8_t* labels, int32_t N, int64_t HW, int32_t C,
                            int32_t square_in_union, const float* partial, int32_t blocks_per_sample, float smooth,
                            int32_t mean, void* dlogits, int32_t ldg, float* loss_partial, float grad_scale,
                            void* stream) {
  B2U_CHECK_ARG(logits && labels && partial && loss_partial && N > 0 && N <= 65535 && HW > 0 && blocks_per_sample > 0,
                "dice_bwd: bad argument");
  B2U_CHECK_ARG(C >= 1 && C <= 32 && C <= ld && (!dlogits || (ldg >= C && ldg % 8 == 0)),
                "dice_bwd: C=%d ld=%d ldg=%d unsupported (ldg must be a multiple of 8)", C, ld, ldg);
  cudaStream_t st = (cudaStream_t)stream;
  const float r = mean ? (float)((double)grad_scale / ((double)N * C)) : grad_scale;
  // loss only (validation): one block per sample folds the statistics
  const dim3 grid(dlogits ? blocks_per_sample : 1, N);
  if (C <= 8)
    launch_k(dice_bwd_kernel<8>, grid, dim3(256), 0, st, logits, ld, labels, (long long)HW, C, square_in_union, partial,
             blocks_per_sample, smooth, r, (bf)dlogits, ldg, loss_partial);
  else
    launch_k(dice_bwd_kernel<32>, grid, dim3(256), 0, st, logits, ld, labels, (long long)HW, C, square_in_union, partial,
             blocks_per_sample, smooth, r, (bf)dlogits, ldg, loss_partial);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_regression_sums(const float* pred, int32_t ld, const float* target, int64_t P, double* partial,
                                   int32_t rows, double* sums, uint32_t* ticket, void* stream) {
  B2U_CHECK_ARG(pred && target && partial && sums && ticket && rows > 0 && P > 0 && ld >= 1, "regression_sums: bad argument");
  launch_k(regression_sums_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, pred, ld, target, (long long)P, partial, sums,
           ticket);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_dice_counts(const float* logits, int32_t ld, const uint8_t* labels, int64_t P, int32_t C,
                               uint64_t* counts, void* stream) {
  B2U_CHECK_ARG(logits && labels && counts && P > 0 && C >= 1 && C <= 32 && C <= ld, "dice_counts: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 8)
    launch_k(dice_counts_kernel<8>, dim3(grid_for(P, 256)), dim3(256), 0, st, logits, ld, labels, (long long)P, C,
             (unsigned long long*)counts);
  else
    launch_k(dice_counts_kernel<32>, dim3(grid_for(P, 256)), dim3(256), 0, st, logits, ld, labels, (long long)P, C,
             (unsigned long long*)counts);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_cast_f32_bf16(const float* x, void* y, int64_t n, void* stream) {
  B2U_CHECK_ARG(x && y && n > 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0,
                "cast_f32_bf16: null / misaligned argument (fp32 range 16-byte, bf16 range 8-byte aligned)");
  launch_k(cast_f32_bf16_kernel, dim3(grid_for(n / 4 + 1, 256)), dim3(256), 0, (cudaStream_t)stream, x, (bf)y, (long long)n);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_cast_bf16_f32(const void* x, float* y, int64_t n, void* stream) {
  B2U_CHECK_ARG(x && y && n > 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0,
                "cast_bf16_f32: null / misaligned argument (fp32 range 16-byte, bf16 range 8-byte aligned)");
  launch_k(cast_bf16_f32_kernel, dim3(grid_for(n / 4 + 1, 256)), dim3(256), 0, (cudaStream_t)stream, (cbf)x, y, (long long)n);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_sgd_step(float* p, const float* g, int64_t n, float lr, float grad_scale, void* stream) {
  B2U_CHECK_ARG(p && g && n > 0, "sgd_step: bad argument");
  launch_k(sgd_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, p, g, n, lr, grad_scale);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_adam_step(float* p, const float* g, float* m, float* v, int64_t n, const int64_t* seg_end,
                             const float* seg_lr, const float* seg_wd, int32_t nseg, const float* hyper,
                             void* stream) {
  B2U_CHECK_ARG(p && g && m && v && n > 0 && seg_end && seg_lr && seg_wd && nseg > 0 && hyper,
                "adam_step: bad argument");
  launch_k(adam_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, n, (const long long*)seg_end, seg_lr,
                                                                  seg_wd, nseg, hyper);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

static int stitch_accumulate_impl(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                                  const int32_t* y0, const int32_t* x0, const int32_t* sel, int32_t n_sel, float* acc,
                                  uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off, int64_t x_off, float quant,
                                  int raw, void* stream, const int32_t* n_sel_dev = nullptr) {
  B2U_CHECK_ARG(logits && y0 && x0 && acc && cnt && C >= 1 && C <= 32 && C <= ld, "stitch_accumulate: bad argument");
  const int nt = sel ? n_sel : T;
  if (nt <= 0) return B2U_OK;
  const long long items = (long long)nt * th * tw;
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 8)
    launch_k(stitch_accumulate_kernel<8>, dim3(grid_for(items, 256)), dim3(256), 0, st, logits, ld, C, T, th, tw, y0, x0,
             sel, n_sel, acc, cnt, Y, X, y_off, x_off, quant, raw, n_sel_dev);
  else
    launch_k(stitch_accumulate_kernel<32>, dim3(grid_for(items, 256)), dim3(256), 0, st, logits, ld, C, T, th, tw, y0, x0,
             sel, n_sel, acc, cnt, Y, X, y_off, x_off, quant, raw, n_sel_dev);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_stitch_accumulate(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                                     const int32_t* y0, const int32_t* x0, const int32_t* sel, int32_t n_sel,
                                     float* acc, uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off, int64_t x_off,
                                     void* stream) {
  return stitch_accumulate_impl(logits, ld, C, T, th, tw, y0, x0, sel, n_sel, acc, cnt, Y, X, y_off, x_off, 0.f, 0, stream);
}

extern "C" int b2u_stitch_accumulate_dev(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                                         const int32_t* y0, const int32_t* x0, const int32_t* sel,
                                         const int32_t* n_sel_dev, int32_t max_sel, int32_t mode, float* acc,
                                         uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off, int64_t x_off,
                                         void* stream) {
  B2U_CHECK_ARG(sel && n_sel_dev && max_sel > 0 && mode >= 0 && mode <= 2, "stitch_accumulate_dev: bad argument");
  return stitch_accumulate_impl(logits, ld, C, T, th, tw, y0, x0, sel, max_sel, acc, cnt, Y, X, y_off, x_off,
                                mode == 1 ? 31.f : 0.f, mode == 2 ? 1 : 0, stream, n_sel_dev);
}

extern "C" int b2u_stitch_accumulate_raw(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                                         const int32_t* y0, const int32_t* x0, const int32_t* sel, int32_t n_sel,
                                         float* acc, uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off, int64_t x_off,
                                         void* stream) {
  return stitch_accumulate_impl(logits, ld, C, T, th, tw, y0, x0, sel, n_sel, acc, cnt, Y, X, y_off, x_off, 0.f, 1, stream);
}

extern "C" int b2u_stitch_finalize_mean(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X,
                                        float nodata, float* out, void* stream) {
  B2U_CHECK_ARG(acc && cnt && out && C >= 1, "stitch_finalize_mean: bad argument");
  launch_k(stitch_finalize_mean_kernel, dim3(grid_for(Y * X, 256)), dim3(256), 0, (cudaStream_t)stream, acc, cnt, C, (long long)(Y * X),
           nodata, out);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_stitch_accumulate_q31(const float* logits, int32_t ld, int32_t C, int32_t T, int32_t th, int32_t tw,
                                         const int32_t* y0, const int32_t* x0, const int32_t* sel, int32_t n_sel,
                                         float* acc, uint8_t* cnt, int64_t Y, int64_t X, int64_t y_off, int64_t x_off,
                                         void* stream) {
  return stitch_accumulate_impl(logits, ld, C, T, th, tw, y0, x0, sel, n_sel, acc, cnt, Y, X, y_off, x_off, 31.f, 0, stream);
}

extern "C" int b2u_stitch_finalize(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X, uint8_t* mask,
                                   void* stream) {
  B2U_CHECK_ARG(acc && cnt && mask && C >= 1, "stitch_finalize: bad argument");
  launch_k(stitch_finalize_kernel, dim3(grid_for(Y * X, 256)), dim3(256), 0, (cudaStream_t)stream, acc, cnt, C, Y * X, mask, 0);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_stitch_finalize_q31(const float* acc, const uint8_t* cnt, int32_t C, int64_t Y, int64_t X,
                                       uint8_t* mask, void* stream) {
  B2U_CHECK_ARG(acc && cnt && mask && C >= 1, "stitch_finalize_q31: bad argument");
  launch_k(stitch_finalize_kernel, dim3(grid_for(Y * X, 256)), dim3(256), 0, (cudaStream_t)stream, acc, cnt, C, Y * X, mask, 1);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_softmax_nchw(const float* logits, int32_t ld, int32_t C, int64_t tiles, int32_t H, int32_t W,
                                float* probs, uint8_t* argmax, void* stream) {
  B2U_CHECK_ARG(logits && C >= 1 && C <= 32 && C <= ld, "softmax_nchw: bad argument");
  const long long items = tiles * H * W;
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 8)
    launch_k(softmax_nchw_kernel<8>, dim3(grid_for(items, 256)), dim3(256), 0, st, logits, ld, C, tiles, H, W, probs, argmax);
  else
    launch_k(softmax_nchw_kernel<32>, dim3(grid_for(items, 256)), dim3(256), 0, st, logits, ld, C, tiles, H, W, probs, argmax);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}

extern "C" int b2u_confusion_counts(const uint8_t* pred, int64_t pred_pitch, int64_t pred_stride, const uint8_t* truth,
                                    int64_t truth_pitch, int64_t truth_stride, int32_t T, int32_t H, int32_t W, int32_t C,
                                    uint64_t* joint, uint32_t* tile_hist, uint64_t* skipped, void* stream) {
  B2U_CHECK_ARG(pred && truth && joint && skipped, "confusion_counts: null argument");
  B2U_CHECK_ARG(T >= 1 && T <= 65535 && H >= 1 && W >= 1 && C >= 1 && C <= 32,
                "confusion_counts: T=%d H=%d W=%d C=%d out of range", T, H, W, C);
  B2U_CHECK_ARG(pred_pitch >= W && truth_pitch >= W &&
                (T == 1 || (pred_stride >= pred_pitch * (H - 1) + W && truth_stride >= truth_pitch * (H - 1) + W)),
                "confusion_counts: pitches %lld / %lld or image strides %lld / %lld too small for %d x %d",
                (long long)pred_pitch, (long long)truth_pitch, (long long)pred_stride, (long long)truth_stride, H, W);
  B2U_CHECK_ARG(!tile_hist || (long long)H * W <= 0xffffffffll, "confusion_counts: %d x %d images overflow tile_hist", H, W);
  // about eight blocks per SM over all images; rows per block a multiple of the 8 warps, and a block's counts stay below
  // 2^31 so that its 32-bit shared counters cannot overflow
  long long gx = std::max(1ll, ((long long)sm_count() * 8 + T - 1) / T);
  long long rows = (H + gx - 1) / gx;
  rows = std::min((rows + 7) / 8 * 8, std::max(1ll, ((1ll << 31) - 1) / W));
  gx = (H + rows - 1) / rows;
  const cudaStream_t st = (cudaStream_t)stream;
  if (C <= 4)
    launch_k(confusion_counts_kernel<true>, dim3((unsigned)gx, T), dim3(256), 0, st, pred, (long long)pred_pitch,
             (long long)pred_stride, truth, (long long)truth_pitch, (long long)truth_stride, H, W, C, (int)rows,
             (unsigned long long*)joint, tile_hist, (unsigned long long*)skipped);
  else
    launch_k(confusion_counts_kernel<false>, dim3((unsigned)gx, T), dim3(256), 0, st, pred, (long long)pred_pitch,
             (long long)pred_stride, truth, (long long)truth_pitch, (long long)truth_stride, H, W, C, (int)rows,
             (unsigned long long*)joint, tile_hist, (unsigned long long*)skipped);
  B2U_LAUNCH_CHECK();
  return B2U_OK;
}
