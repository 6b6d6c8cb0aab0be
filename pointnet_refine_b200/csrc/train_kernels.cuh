// CUDA-core kernels of the train-mode path (batch-statistic BatchNorm forward and the hand-written
// backward).  All GEMMs of that path (forward, dgrad, wgrad) go through the tcgen05 pair kernels; these
// kernels are the HBM-bound glue: statistics, normalisation, gate, masks, small reductions.
// Reference semantics: torch.nn.BatchNorm1d in training mode (biased variance for normalisation, unbiased
// for the running update, momentum 0.1) as used by src/model.py:16-20,25,43-51.
#pragma once
#include <cuda_bf16.h>

#include "ptx.cuh"

namespace lrn {

__device__ __forceinline__ float bf2f(__nv_bfloat16 v) { return __bfloat162float(v); }

// dst (bf16, row pitch ld) <- src fp32 (rows x cols), optionally transposed.  dst is zero-filled beforehand.
__global__ void pack_bf16_kernel(const float* __restrict__ src, int rows, int cols, __nv_bfloat16* __restrict__ dst,
                                 long long ld, int transpose) {
  const long long total = static_cast<long long>(rows) * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<long long>(r) * cols);
    dst[transpose ? c * ld + r : r * ld + c] = __float2bfloat16_rn(src[i]);
  }
}

// conv1 pre-activation U1 = W1 x + b1 (raw fp32 point, no BatchNorm yet) and gate hidden H = relu(wg1 I + bg1).
// 16 threads per point, 4 + 4 channels each (same mapping as point_embed_kernel).
__global__ void __launch_bounds__(256)
train_embed_kernel(const float4* __restrict__ ctx, long long rows, const float* __restrict__ w1,
                   const float* __restrict__ b1, const float* __restrict__ wg1, const float* __restrict__ bg1,
                   __nv_bfloat16* __restrict__ U, long long ldu, __nv_bfloat16* __restrict__ X, long long ldx) {
  const int sub = threadIdx.x & 15;
  float4 wr[4];
  float br[4], gw[4], gb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    wr[j] = reinterpret_cast<const float4*>(w1)[4 * sub + j];
    br[j] = b1[4 * sub + j];
    gw[j] = wg1[4 * sub + j];
    gb[j] = bg1[4 * sub + j];
  }
  const long long ppb = blockDim.x / 16;
  for (long long pt = blockIdx.x * ppb + (threadIdx.x >> 4); pt < rows; pt += gridDim.x * ppb) {
    const float4 x = __ldg(ctx + pt);
    float u[4], h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      u[j] = fmaf(wr[j].x, x.x, fmaf(wr[j].y, x.y, fmaf(wr[j].z, x.z, fmaf(wr[j].w, x.w, br[j]))));
      h[j] = fmaxf(fmaf(gw[j], x.w, gb[j]), 0.f);
    }
    *reinterpret_cast<uint2*>(U + pt * ldu + 4 * sub) = make_uint2(ptx::pack_bf16x2(u[0], u[1]), ptx::pack_bf16x2(u[2], u[3]));
    *reinterpret_cast<uint2*>(X + pt * ldx + 1984 + 4 * sub) =
        make_uint2(ptx::pack_bf16x2(h[0], h[1]), ptx::pack_bf16x2(h[2], h[3]));
  }
}

// Per-column sum and sum of squares of a bf16 (rows x C) matrix -> fp32 atomics into sum[C], sumsq[C].
// `shifted`: the sums are taken of (x - K_c) with the pivot K_c = A[0][c] (row 0 of the same column), so that the
// variance E[(x-K)^2] - E[x-K]^2 formed from them does not cancel when |mean| >> std (the naive E[x^2] - mean^2 in
// fp32 loses all digits there); bn_finalize_kernel adds the pivot back.
// Block = 64 columns as 8 channel groups of 8 (one 16-byte load per thread and row: 8 threads cover 128 contiguous bytes)
// x 32 row lanes, two independent loads in flight per thread; grid = (C / 64, row slabs).  Requires a 16-byte aligned base
// and a row pitch that is a multiple of 8 elements.
__global__ void __launch_bounds__(256, 4)
col_stats_kernel(const __nv_bfloat16* __restrict__ A, long long ld, long long rows, float* __restrict__ sum,
                 float* __restrict__ sumsq, int shifted) {
  const int cg = threadIdx.x & 7, lane_r = threadIdx.x >> 3;
  const int c = blockIdx.x * 64 + 8 * cg;
  float piv[8], s[8], q[8];
  {
    uint4 raw = make_uint4(0, 0, 0, 0);
    if (shifted) raw = *reinterpret_cast<const uint4*>(A + c);
    const __nv_bfloat16* pv = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      piv[j] = bf2f(pv[j]);
      s[j] = q[j] = 0.f;
    }
  }
  auto acc = [&](const uint4& raw) {
    const __nv_bfloat16* v = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float f = bf2f(v[j]) - piv[j];
      s[j] += f;
      q[j] = fmaf(f, f, q[j]);
    }
  };
  // four independent 16-byte loads in flight per thread (4 resident blocks x 256 threads: 64 KB per SM on the wire)
  const long long stride = gridDim.y * 32ll;
  long long r = blockIdx.y * 32ll + lane_r;
  for (; r + 3 * stride < rows; r += 4 * stride) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(A + r * ld + c);
    const uint4 v1 = *reinterpret_cast<const uint4*>(A + (r + stride) * ld + c);
    const uint4 v2 = *reinterpret_cast<const uint4*>(A + (r + 2 * stride) * ld + c);
    const uint4 v3 = *reinterpret_cast<const uint4*>(A + (r + 3 * stride) * ld + c);
    acc(v0);
    acc(v1);
    acc(v2);
    acc(v3);
  }
  for (; r < rows; r += stride) acc(*reinterpret_cast<const uint4*>(A + r * ld + c));
  __shared__ float sh[2][32][65];   // [sum | sumsq][row lane][column of the block]
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sh[0][lane_r][8 * cg + j] = s[j];
    sh[1][lane_r][8 * cg + j] = q[j];
  }
  __syncthreads();
  if (threadIdx.x < 128) {  // threads 0..63: sums of the 64 columns, 64..127: sums of squares
    const int which = threadIdx.x >> 6, col = threadIdx.x & 63;
    float t = 0.f;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) t += sh[which][k][col];
    if (which == 0) atomicAdd(sum + blockIdx.x * 64 + col, t);
    else if (sumsq) atomicAdd(sumsq + blockIdx.x * 64 + col, t);
  }
}

// Batch statistics -> mean / rstd, the fused scale/shift of the normalisation, and the running-stat update.
// sum / sumsq are the pivot-shifted sums of col_stats_kernel (pivot_row = row 0 of the matrix they were taken of).
__global__ void bn_finalize_kernel(const float* __restrict__ sum, const float* __restrict__ sumsq,
                                   const __nv_bfloat16* __restrict__ pivot_row, long long rows, int C,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ scale,
                                   float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float n = static_cast<float>(rows);
  const float d = sum[c] / n;                          // mean of (x - pivot)
  const float m = bf2f(pivot_row[c]) + d;
  const float var = fmaxf(sumsq[c] / n - d * d, 0.f);  // biased; shift-invariant
  const float r = rsqrtf(var + eps);
  mean[c] = m;
  rstd[c] = r;
  scale[c] = gamma[c] * r;
  shift[c] = beta[c] - m * gamma[c] * r;
  if (running_mean) {
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * (rows > 1 ? n / (n - 1.f) : 1.f);
  }
}

// X[:, c] = relu(U[:, c] * scale[c] + shift[c]).  Channel-stationary threads: a thread owns 8 channels (its
// scale / shift stay in registers) and walks down the rows; 8 threads cover 128 contiguous bytes of a row.
// grid = (C / 64, row slabs), block = 8 channel groups x 32 row lanes.
__global__ void __launch_bounds__(256, 4)
bn_relu_apply_kernel(const __nv_bfloat16* __restrict__ U, long long ldu, long long rows, int C,
                     const float* __restrict__ scale, const float* __restrict__ shift, __nv_bfloat16* __restrict__ X,
                     long long ldx) {
  const int c0 = blockIdx.x * 64 + (threadIdx.x & 7) * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c0 + j]; sh[j] = shift[c0 + j]; }
  auto apply = [&](const uint4& raw, long long r) {
    const __nv_bfloat16* u = reinterpret_cast<const __nv_bfloat16*>(&raw);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(bf2f(u[j]), sc[j], sh[j]), 0.f);
    *reinterpret_cast<uint4*>(X + r * ldx + c0) =
        make_uint4(ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]), ptx::pack_bf16x2(v[4], v[5]),
                   ptx::pack_bf16x2(v[6], v[7]));
  };
  const long long stride = gridDim.y * 32ll;
  long long r = blockIdx.y * 32ll + (threadIdx.x >> 3);
  for (; r + 3 * stride < rows; r += 4 * stride) {   // four loads in flight per thread
    const uint4 v0 = *reinterpret_cast<const uint4*>(U + r * ldu + c0);
    const uint4 v1 = *reinterpret_cast<const uint4*>(U + (r + stride) * ldu + c0);
    const uint4 v2 = *reinterpret_cast<const uint4*>(U + (r + 2 * stride) * ldu + c0);
    const uint4 v3 = *reinterpret_cast<const uint4*>(U + (r + 3 * stride) * ldu + c0);
    apply(v0, r);
    apply(v1, r + stride);
    apply(v2, r + 2 * stride);
    apply(v3, r + 3 * stride);
  }
  for (; r < rows; r += stride) apply(*reinterpret_cast<const uint4*>(U + r * ldu + c0), r);
}

__device__ __forceinline__ float sigmoidf_fast(float z) { return __fdividef(1.f, 1.f + __expf(-z)); }

// 16-byte shared-memory read that the compiler may not hoist out of a loop: per-channel constants that are re-read per row
// instead of living in registers (the streaming kernels below trade eight LDS.128 per row for 16 - 24 registers, i.e. for
// a second row of loads in flight at the same occupancy).
__device__ __forceinline__ float4 lds_f4_pinned(const float* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ptx::smem_u32(p)));
  return v;
}


// fused[b, c, n] = relu(Uf[p, c] * scale[c] + shift[c]) * (0.5 + 0.5 * sigmoid(Z[p, c])),  p = b * N + n
// (src/model.py:51,54-55, train mode).  32 points x 32 channels per block, transposed through shared memory so
// both the point-major reads and the channel-major (B,1024,N) writes are coalesced.
__global__ void __launch_bounds__(256)
fusion_gate_fwd_kernel(const __nv_bfloat16* __restrict__ Uf, long long ldu, const __nv_bfloat16* __restrict__ Z,
                       long long ldz, long long rows, int npts, const float* __restrict__ scale,
                       const float* __restrict__ shift, float* __restrict__ fused) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long p0 = blockIdx.x * 32ll;
  const int c0 = blockIdx.y * 32;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long p = p0 + ty + 8 * k;
    float v = 0.f;
    if (p < rows) {
      const int c = c0 + tx;
      const float y = fmaxf(fmaf(bf2f(Uf[p * ldu + c]), scale[c], shift[c]), 0.f);
      v = y * (0.5f + 0.5f * sigmoidf_fast(bf2f(Z[p * ldz + c])));
    }
    tile[ty + 8 * k][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c0 + ty + 8 * k;
    const long long p = p0 + tx;
    if (p < rows) {
      const unsigned b = static_cast<unsigned>(p) / static_cast<unsigned>(npts), n = static_cast<unsigned>(p) - b * npts;
      fused[(static_cast<long long>(b) * 1024 + c) * npts + n] = tile[tx][ty + 8 * k];
    }
  }
}

// Dual pooling of the train-mode output (src/model.py:58-60): one warp per (segment, channel) row of fused (B,1024,N):
// global_feat[b, c] = max_n, global_feat[b, 1024 + c] = mean_n, argmax[b, c] = first maximal n (torch.max's rule) -
// the index the backward scatters the max gradient to.
__global__ void __launch_bounds__(256)
pool_rows_kernel(const float* __restrict__ fused, long long rows /* B * 1024 */, int npts, float* __restrict__ global_feat,
                 long long* __restrict__ argmax) {
  const int lane = threadIdx.x & 31;
  const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long r = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps) {
    const float* row = fused + r * npts;
    float best = -INFINITY, sum = 0.f;
    int arg = 0x7FFFFFFF;
    for (int n = lane; n < npts; n += 32) {
      const float v = row[n];
      sum += v;
      if (v > best) {   // strictly greater: the first index wins inside a lane
        best = v;
        arg = n;
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if (ob > best || (ob == best && oa < arg)) {
        best = ob;
        arg = oa;
      }
    }
    if (lane == 0) {
      const long long b = r >> 10, c = r & 1023;
      global_feat[b * 2048 + c] = best;
      global_feat[b * 2048 + 1024 + c] = sum / static_cast<float>(npts);
      argmax[r] = arg;
    }
  }
}

// Point-major variants (no layout change): fused_pm[p, c] bf16, channel-stationary threads like bn_relu_apply_kernel.
__global__ void __launch_bounds__(256, 4)
fusion_gate_fwd_pm_kernel(const __nv_bfloat16* __restrict__ Uf, long long ldu, const __nv_bfloat16* __restrict__ Z,
                          long long ldz, long long rows, const float* __restrict__ scale, const float* __restrict__ shift,
                          __nv_bfloat16* __restrict__ fused_pm) {
  const int c0 = blockIdx.x * 64 + (threadIdx.x & 7) * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c0 + j]; sh[j] = shift[c0 + j]; }
  for (long long r = blockIdx.y * 32ll + (threadIdx.x >> 3); r < rows; r += gridDim.y * 32ll) {
    const uint4 ru = *reinterpret_cast<const uint4*>(Uf + r * ldu + c0);
    const uint4 rz = *reinterpret_cast<const uint4*>(Z + r * ldz + c0);
    const __nv_bfloat16 *u = reinterpret_cast<const __nv_bfloat16*>(&ru), *z = reinterpret_cast<const __nv_bfloat16*>(&rz);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j)
      v[j] = fmaxf(fmaf(bf2f(u[j]), sc[j], sh[j]), 0.f) * (0.5f + 0.5f * sigmoidf_fast(bf2f(z[j])));
    *reinterpret_cast<uint4*>(fused_pm + r * 1024 + c0) =
        make_uint4(ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]), ptx::pack_bf16x2(v[4], v[5]),
                   ptx::pack_bf16x2(v[6], v[7]));
  }
}

// Besides dY / dZ it accumulates the three column sums the next steps need, from the rounded values it stores - the
// fusion BatchNorm backward's S1 = sum dY, S2 = sum dY * xhat (xhat = (Uf - mean) * rstd) and Sz = sum dZ (the gate
// layer 2 bias gradient) - so neither dY nor dZ is read again for a reduction pass.
__global__ void __launch_bounds__(256, 3)
fusion_gate_bwd_pm_kernel(const __nv_bfloat16* __restrict__ dfused_pm, const __nv_bfloat16* __restrict__ Uf, long long ldu,
                          const __nv_bfloat16* __restrict__ Z, long long ldz, long long rows,
                          const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ mean,
                          const float* __restrict__ rstd, __nv_bfloat16* __restrict__ dY, __nv_bfloat16* __restrict__ dZ,
                          long long ldd, float* __restrict__ S1, float* __restrict__ S2, float* __restrict__ Sz) {
  const int cg = threadIdx.x & 7, lane_r = threadIdx.x >> 3;
  const int c0 = blockIdx.x * 64 + cg * 8;
  float sc[8], sh[8], m[8], s1[8], s2[8], sz[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[c0 + j];
    sh[j] = shift[c0 + j];
    m[j] = mean[c0 + j];
    s1[j] = s2[j] = sz[j] = 0.f;
  }
  for (long long r = blockIdx.y * 32ll + lane_r; r < rows; r += gridDim.y * 32ll) {
    const uint4 rd = *reinterpret_cast<const uint4*>(dfused_pm + r * 1024 + c0);
    const uint4 ru = *reinterpret_cast<const uint4*>(Uf + r * ldu + c0);
    const uint4 rz = *reinterpret_cast<const uint4*>(Z + r * ldz + c0);
    const __nv_bfloat16 *d = reinterpret_cast<const __nv_bfloat16*>(&rd), *u = reinterpret_cast<const __nv_bfloat16*>(&ru),
                        *z = reinterpret_cast<const __nv_bfloat16*>(&rz);
    __align__(16) __nv_bfloat16 a[8], b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float df = bf2f(d[j]);
      const float uj = bf2f(u[j]);
      const float y0 = fmaf(uj, sc[j], sh[j]);
      const float g = sigmoidf_fast(bf2f(z[j]));
      a[j] = __float2bfloat16_rn(y0 > 0.f ? df * (0.5f + 0.5f * g) : 0.f);
      b[j] = __float2bfloat16_rn(df * fmaxf(y0, 0.f) * 0.5f * g * (1.f - g));
      const float af = bf2f(a[j]);
      s1[j] += af;
      s2[j] = fmaf(af, uj - m[j], s2[j]);      // rstd is applied once per block below
      sz[j] += bf2f(b[j]);
    }
    *reinterpret_cast<uint4*>(dY + r * ldd + c0) = *reinterpret_cast<const uint4*>(a);
    *reinterpret_cast<uint4*>(dZ + r * ldd + c0) = *reinterpret_cast<const uint4*>(b);
  }
  __shared__ float shm[3][32][65];   // [S1 | S2 | Sz][row lane][column of the block]
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    shm[0][lane_r][8 * cg + j] = s1[j];
    shm[1][lane_r][8 * cg + j] = s2[j];
    shm[2][lane_r][8 * cg + j] = sz[j];
  }
  __syncthreads();
  if (threadIdx.x < 192) {
    const int which = threadIdx.x >> 6, col = threadIdx.x & 63;
    float t = 0.f;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) t += shm[which][k][col];
    if (which == 1) t *= rstd[blockIdx.x * 64 + col];
    atomicAdd((which == 0 ? S1 : which == 1 ? S2 : Sz) + blockIdx.x * 64 + col, t);
  }
}

// Backward of the gate / ReLU at the fused output: with y0 = Uf*scale+shift, y = relu(y0), g = sigmoid(Z):
//   dY[p,c] = dF * (0.5 + 0.5 g) * [y0 > 0]      (gradient w.r.t. the BatchNorm output)
//   dZ[p,c] = dF * y * 0.5 * g * (1 - g)         (gradient w.r.t. the gate pre-activation)
// The gradient of the pooled features is folded in here (hand-written backward of src/model.py:58-60): the max gradient
// is scattered to its argmax point, the mean gradient spread as 1/N - `dfused` may then be null (pooled loss only),
// no dense (B,1024,N) gradient is ever built for the pooling.
__global__ void __launch_bounds__(256)
fusion_gate_bwd_kernel(const float* __restrict__ dfused, const float* __restrict__ dgf, const long long* __restrict__ argmax,
                       const __nv_bfloat16* __restrict__ Uf, long long ldu,
                       const __nv_bfloat16* __restrict__ Z, long long ldz, long long rows, int npts,
                       const float* __restrict__ scale, const float* __restrict__ shift, __nv_bfloat16* __restrict__ dY,
                       __nv_bfloat16* __restrict__ dZ, long long ldd) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long p0 = blockIdx.x * 32ll;
  const int c0 = blockIdx.y * 32;
#pragma unroll
  for (int k = 0; k < 4; ++k) {  // coalesced along n: tile[c][p]
    const int c = c0 + ty + 8 * k;
    const long long p = p0 + tx;
    float v = 0.f;
    if (p < rows) {
      const unsigned b = static_cast<unsigned>(p) / static_cast<unsigned>(npts), n = static_cast<unsigned>(p) - b * npts;
      if (dfused) v = dfused[(static_cast<long long>(b) * 1024 + c) * npts + n];
      if (dgf) {
        v += dgf[static_cast<long long>(b) * 2048 + 1024 + c] / static_cast<float>(npts);
        if (argmax[static_cast<long long>(b) * 1024 + c] == n) v += dgf[static_cast<long long>(b) * 2048 + c];
      }
    }
    tile[ty + 8 * k][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long p = p0 + ty + 8 * k;
    if (p < rows) {
      const int c = c0 + tx;
      const float df = tile[tx][ty + 8 * k];
      const float y0 = fmaf(bf2f(Uf[p * ldu + c]), scale[c], shift[c]);
      const float g = sigmoidf_fast(bf2f(Z[p * ldz + c]));
      dY[p * ldd + c] = __float2bfloat16_rn(y0 > 0.f ? df * (0.5f + 0.5f * g) : 0.f);
      dZ[p * ldd + c] = __float2bfloat16_rn(df * fmaxf(y0, 0.f) * 0.5f * g * (1.f - g));
    }
  }
}

// BatchNorm backward, pass 1: S1[c] = sum_p dY, S2[c] = sum_p dY * xhat, where
//   dY = (d1 + d2) * [scale * U + shift > 0]   (d2 optional: a second gradient source; the ReLU mask is re-derived from
//        the pre-activation U, which this pass reads anyway, with the forward's own scale / shift - the same fmaf whose
//        sign decided the stored activation - instead of reading the activation matrix as a fourth stream; msc = null: no ReLU)
//   xhat = (U - mean) * rstd
// Block = 64 columns as 8 channel groups of 8 (16-byte loads) x 32 row lanes; grid = (C / 64, row slabs).
// The thread accumulates A = sum dY and T = sum dY * (U - mean); S2 = rstd * T is formed once per block (rstd is not held
// per thread: 3 resident blocks, and two rows = up to six 16-byte loads in flight per thread).
__global__ void __launch_bounds__(256, 3)
bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ d1, long long ld1, const __nv_bfloat16* __restrict__ d2,
                     long long ld2, const float* __restrict__ msc, const float* __restrict__ msh,
                     const __nv_bfloat16* __restrict__ U, long long ldu, long long rows, const float* __restrict__ mean,
                     const float* __restrict__ rstd, float* __restrict__ S1, float* __restrict__ S2) {
  const int cg = threadIdx.x & 7, lane_r = threadIdx.x >> 3;
  const int c = blockIdx.x * 64 + 8 * cg;
  float sc[8], sh[8], m[8], a[8], t[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = msc ? msc[c + j] : 0.f;
    sh[j] = msc ? msh[c + j] : 0.f;
    m[j] = mean[c + j];
    a[j] = t[j] = 0.f;
  }
  auto acc = [&](const uint4& r1, const uint4& r2, const uint4& ru) {
    const __nv_bfloat16 *p1 = reinterpret_cast<const __nv_bfloat16*>(&r1), *p2 = reinterpret_cast<const __nv_bfloat16*>(&r2),
                        *pu = reinterpret_cast<const __nv_bfloat16*>(&ru);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float d = bf2f(p1[j]);
      const float u = bf2f(pu[j]);
      if (d2) d += bf2f(p2[j]);
      if (msc && !(fmaf(u, sc[j], sh[j]) > 0.f)) d = 0.f;
      a[j] += d;
      t[j] = fmaf(d, u - m[j], t[j]);
    }
  };
  const uint4 zero = make_uint4(0, 0, 0, 0);
  const long long stride = gridDim.y * 32ll;
  long long r = blockIdx.y * 32ll + lane_r;
  for (; r + stride < rows; r += 2 * stride) {
    const long long rb = r + stride;
    const uint4 a1 = *reinterpret_cast<const uint4*>(d1 + r * ld1 + c);
    const uint4 au = *reinterpret_cast<const uint4*>(U + r * ldu + c);
    const uint4 b1 = *reinterpret_cast<const uint4*>(d1 + rb * ld1 + c);
    const uint4 bu = *reinterpret_cast<const uint4*>(U + rb * ldu + c);
    uint4 a2 = zero, b2 = zero;
    if (d2) {
      a2 = *reinterpret_cast<const uint4*>(d2 + r * ld2 + c);
      b2 = *reinterpret_cast<const uint4*>(d2 + rb * ld2 + c);
    }
    acc(a1, a2, au);
    acc(b1, b2, bu);
  }
  if (r < rows) {
    const uint4 a1 = *reinterpret_cast<const uint4*>(d1 + r * ld1 + c);
    const uint4 au = *reinterpret_cast<const uint4*>(U + r * ldu + c);
    const uint4 a2 = d2 ? *reinterpret_cast<const uint4*>(d2 + r * ld2 + c) : zero;
    acc(a1, a2, au);
  }
  __shared__ float shm[2][32][65];   // [A | T][row lane][column of the block]
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    shm[0][lane_r][8 * cg + j] = a[j];
    shm[1][lane_r][8 * cg + j] = t[j];
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int col = threadIdx.x, ch = blockIdx.x * 64 + col;
    float sa = 0.f, st = 0.f;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      sa += shm[0][k][col];
      st += shm[1][k][col];
    }
    atomicAdd(S1 + ch, sa);
    atomicAdd(S2 + ch, rstd[ch] * st);
  }
}

// BatchNorm backward, pass 2: dU = gamma * rstd * (dY - S1/P - xhat * S2/P) = A_c dY + B_c U + C_c with per-channel
// coefficients kept in registers (channel-stationary threads as in bn_relu_apply_kernel).
// d1 may alias dU (in place): every element is read before it is written by the same thread.
__global__ void __launch_bounds__(256, 3)
bn_bwd_apply_kernel(const __nv_bfloat16* d1, long long ld1, const __nv_bfloat16* __restrict__ d2, long long ld2,
                    const float* __restrict__ msc, const float* __restrict__ msh, const __nv_bfloat16* __restrict__ U,
                    long long ldu, long long rows, int C, const float* __restrict__ mean,
                    const float* __restrict__ rstd, const float* __restrict__ gamma, const float* __restrict__ S1,
                    const float* __restrict__ S2, __nv_bfloat16* dU, long long ldo) {
  __shared__ __align__(16) float smask[2][64];   // the ReLU mask's scale / shift of the block's 64 channels
  if (threadIdx.x < 128) {
    const int which = threadIdx.x >> 6, col = threadIdx.x & 63;
    smask[which][col] = msc ? (which ? msh : msc)[blockIdx.x * 64 + col] : 0.f;
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;
  const int c0 = blockIdx.x * 64 + cg * 8;
  const float inv_n = 1.f / static_cast<float>(rows);
  float A[8], Bc[8], Cc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = c0 + j;
    const float gr = gamma[c] * rstd[c];
    A[j] = gr;
    Bc[j] = -gr * rstd[c] * S2[c] * inv_n;
    Cc[j] = -gr * S1[c] * inv_n - Bc[j] * mean[c];
  }
  auto apply = [&](const uint4& r1, const uint4& r2, const uint4& ru, long long r) {
    const __nv_bfloat16 *p1 = reinterpret_cast<const __nv_bfloat16*>(&r1), *p2 = reinterpret_cast<const __nv_bfloat16*>(&r2),
                        *pu = reinterpret_cast<const __nv_bfloat16*>(&ru);
    float v[8];
#pragma unroll
    for (int hq = 0; hq < 2; ++hq) {
      float sc[4] = {0.f, 0.f, 0.f, 0.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
      if (msc) {
        const float4 a = lds_f4_pinned(&smask[0][8 * cg + 4 * hq]), b = lds_f4_pinned(&smask[1][8 * cg + 4 * hq]);
        sc[0] = a.x; sc[1] = a.y; sc[2] = a.z; sc[3] = a.w;
        sh[0] = b.x; sh[1] = b.y; sh[2] = b.z; sh[3] = b.w;
      }
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int j = 4 * hq + jj;
        float d = bf2f(p1[j]);
        const float u = bf2f(pu[j]);
        if (d2) d += bf2f(p2[j]);
        if (msc && !(fmaf(u, sc[jj], sh[jj]) > 0.f)) d = 0.f;   // ReLU mask from the pre-activation (see bn_bwd_reduce_kernel)
        v[j] = fmaf(A[j], d, fmaf(Bc[j], u, Cc[j]));
      }
    }
    *reinterpret_cast<uint4*>(dU + r * ldo + c0) =
        make_uint4(ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]), ptx::pack_bf16x2(v[4], v[5]),
                   ptx::pack_bf16x2(v[6], v[7]));
  };
  // two rows = up to six 16-byte loads in flight per thread at 3 resident blocks (the mask constants come from shared
  // memory per row, so the 24 BatchNorm coefficients + two rows of loads fit without spills); both rows are read before
  // either is written (d1 may alias dU)
  const uint4 zero = make_uint4(0, 0, 0, 0);
  const long long stride = gridDim.y * 32ll;
  long long r = blockIdx.y * 32ll + (threadIdx.x >> 3);
  for (; r + stride < rows; r += 2 * stride) {
    const long long rb = r + stride;
    const uint4 a1 = *reinterpret_cast<const uint4*>(d1 + r * ld1 + c0);
    const uint4 au = *reinterpret_cast<const uint4*>(U + r * ldu + c0);
    const uint4 b1 = *reinterpret_cast<const uint4*>(d1 + rb * ld1 + c0);
    const uint4 bu = *reinterpret_cast<const uint4*>(U + rb * ldu + c0);
    uint4 a2 = zero, b2 = zero;
    if (d2) {
      a2 = *reinterpret_cast<const uint4*>(d2 + r * ld2 + c0);
      b2 = *reinterpret_cast<const uint4*>(d2 + rb * ld2 + c0);
    }
    apply(a1, a2, au, r);
    apply(b1, b2, bu, rb);
  }
  if (r < rows) {
    const uint4 a1 = *reinterpret_cast<const uint4*>(d1 + r * ld1 + c0);
    const uint4 au = *reinterpret_cast<const uint4*>(U + r * ldu + c0);
    const uint4 a2 = d2 ? *reinterpret_cast<const uint4*>(d2 + r * ld2 + c0) : zero;
    apply(a1, a2, au, r);
  }
}

// conv1 / gate layer 1 parameter gradients (K = 4 resp. 1: plain reductions over the points):
//   dW1[c, :] = sum_p dU1[p, c] * x[p, :]    db1[c] = sum_p dU1[p, c]
//   dwg1[c]   = sum_p dH[p, c] * [H > 0] * I  dbg1[c] = sum_p dH[p, c] * [H > 0]
__global__ void __launch_bounds__(256)
conv1_gate1_bwd_kernel(const float4* __restrict__ ctx, long long rows, const __nv_bfloat16* __restrict__ dU1,
                       long long ldu, const __nv_bfloat16* __restrict__ dH, long long ldh,
                       const __nv_bfloat16* __restrict__ H, long long ldx, float* __restrict__ dW1,
                       float* __restrict__ db1, float* __restrict__ dwg1, float* __restrict__ dbg1) {
  const int c = threadIdx.x & 63, lane_r = threadIdx.x >> 6;
  float a[4] = {0.f, 0.f, 0.f, 0.f}, ab = 0.f, g = 0.f, gb = 0.f;
  for (long long r = blockIdx.x * 4ll + lane_r; r < rows; r += gridDim.x * 4ll) {
    const float4 x = __ldg(ctx + r);
    const float du = bf2f(dU1[r * ldu + c]);
    a[0] = fmaf(du, x.x, a[0]);
    a[1] = fmaf(du, x.y, a[1]);
    a[2] = fmaf(du, x.z, a[2]);
    a[3] = fmaf(du, x.w, a[3]);
    ab += du;
    const float dh = bf2f(H[r * ldx + c]) > 0.f ? bf2f(dH[r * ldh + c]) : 0.f;
    g = fmaf(dh, x.w, g);
    gb += dh;
  }
  __shared__ float sh[7][4][64];
  sh[0][lane_r][c] = a[0]; sh[1][lane_r][c] = a[1]; sh[2][lane_r][c] = a[2]; sh[3][lane_r][c] = a[3];
  sh[4][lane_r][c] = ab;   sh[5][lane_r][c] = g;    sh[6][lane_r][c] = gb;
  __syncthreads();
  if (lane_r == 0) {
    float t[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) t[k] = sh[k][0][c] + sh[k][1][c] + sh[k][2][c] + sh[k][3][c];
    atomicAdd(dW1 + 4 * c + 0, t[0]);
    atomicAdd(dW1 + 4 * c + 1, t[1]);
    atomicAdd(dW1 + 4 * c + 2, t[2]);
    atomicAdd(dW1 + 4 * c + 3, t[3]);
    atomicAdd(db1 + c, t[4]);
    atomicAdd(dwg1 + c, t[5]);
    atomicAdd(dbg1 + c, t[6]);
  }
}

// out[r, c] = src[r * ld + c0 + c] for c < cols  (fp32 sub-matrix copy: wgrad temporaries -> gradient tensors)
__global__ void copy_submatrix_kernel(const float* __restrict__ src, long long ld, int c0, int rows, int cols,
                                      float* __restrict__ dst) {
  const long long total = static_cast<long long>(rows) * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<long long>(r) * cols);
    dst[i] = src[r * ld + c0 + c];
  }
}

// ---------------------------------------------------------------------------------------------
// Training-loop machinery (SURVEY.md 8f row 4): Adam over one flat parameter buffer and the L1 deep-supervision loss.
// ---------------------------------------------------------------------------------------------
// torch.optim.Adam (train.py:40, no amsgrad), same operation order as its single-tensor path:
//   g += wd * p;  m = m + (1 - b1) (g - m);  v = b2 v + (1 - b2) g g;  p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
// The step count is in device memory (torch.optim.Adam(capturable=True)), so a captured CUDA graph replays the step with
// the right bias corrections.  adam_bump_step_kernel runs first in the stream (step += 1).
__global__ void adam_bump_step_kernel(long long* step) { *step += 1; }

__global__ void __launch_bounds__(256)
adam_step_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                     float lr, float b1, float b2, float eps, float wd, const long long* __restrict__ step) {
  __shared__ float sh[2];
  if (threadIdx.x == 0) {
    const double t = static_cast<double>(*step);
    sh[0] = static_cast<float>(static_cast<double>(lr) / (1.0 - pow(static_cast<double>(b1), t)));
    sh[1] = static_cast<float>(1.0 / sqrt(1.0 - pow(static_cast<double>(b2), t)));
  }
  __syncthreads();
  const float step_size = sh[0], inv_bc2_sqrt = sh[1];
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    float gi = g[i];
    const float pi = p[i];
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    const float mi = fmaf(1.f - b1, gi - m[i], m[i]);
    const float vi = fmaf(1.f - b2, gi * gi, b2 * v[i]);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - step_size * (mi / (sqrtf(vi) * inv_bc2_sqrt + eps));
  }
}

// loss = (1 / L) sum_l mean_i |pred[l][i] - target[i]|   (train.py:63-69, criterion = L1Loss);
// dpred[l][i] = sign(pred[l][i] - target[i]) / (L n)       (0 at equality, like torch)
__global__ void __launch_bounds__(256)
l1_deep_supervision_kernel(const float* __restrict__ pred, const float* __restrict__ target, int L, long long n,
                           float* __restrict__ loss, float* __restrict__ dpred) {
  __shared__ float red[8];
  const float w = 1.f / (static_cast<float>(L) * static_cast<float>(n));
  const long long total = static_cast<long long>(L) * n, stride = static_cast<long long>(gridDim.x) * blockDim.x;
  float acc = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const float d = pred[i] - target[i % n];
    acc += fabsf(d);
    if (dpred) dpred[i] = d > 0.f ? w : (d < 0.f ? -w : 0.f);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(loss, t * w);
  }
}

}  // namespace lrn
