// Per-line preprocessing of a whole scene on the GPU (SURVEY.md section 8f row 3): tube crop, weighted sampling without
// replacement, centroid normalisation, for all lines of a scene in one pass - the work the reference does on the host
// with a KD-tree per line (src/dataset.py:78-130,214-237; inference_whole_scene.py:95-121).
//
// Index work is bit-exact against oracle/scene_oracle.py by construction: distances, weights and keys are fixed
// sequences of IEEE double operations (__dmul_rn / __dadd_rn: no fused multiply-add), the random numbers are a
// counter-based hash of (seed, line, scene index), and the selection is order-independent (top-N keys, sorted).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lrn {
namespace scene {

constexpr int kDense = 200;  // points of the crop polyline (src/dataset.py:217)
constexpr int kLine = 32;    // points of the sampling polyline
constexpr int kLineTile = 256;
constexpr int kSub = 8;                    // the crop polyline is tested in 8 pieces of 25 points, each with its own box
constexpr int kSubLen = kDense / kSub;
constexpr int kBoxFloats = 6 * (1 + kSub);  // per line: whole-line box, then the piece boxes

// ------------------------------------------------------------------------------------------------ RNG contract
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double det_uniform(uint64_t seed, uint64_t line, uint64_t idx) {
  const uint64_t x = seed + 0x9E3779B97F4A7C15ull * (line + 1) + 0xD1B54A32D192ED03ull * (idx + 1);
  return __dmul_rn(__dadd_rn(static_cast<double>(splitmix64(x) >> 11), 0.5), 1.1102230246251565404e-16);  // 2^-53
}
constexpr double kLn2Hi = 6.93147180369123816490e-01, kLn2Lo = 1.90821492927058770002e-10, kInvLn2 = 1.44269504088896338700e+00;

__device__ __forceinline__ double det_exp(double x) {
  const double n = rint(__dmul_rn(x, kInvLn2));
  const double r = __dsub_rn(__dsub_rn(x, __dmul_rn(n, kLn2Hi)), __dmul_rn(n, kLn2Lo));
  const double c[13] = {1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 5040.0, 1.0 / 720.0,
                        1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5, 1.0, 1.0};
  double p = 1.0 / 6227020800.0;
#pragma unroll
  for (int i = 0; i < 13; ++i) p = __dadd_rn(__dmul_rn(p, r), c[i]);
  return ldexp(p, static_cast<int>(n));
}
__device__ __forceinline__ double det_log(double u) {
  int e;
  double m = frexp(u, &e);
  if (m < 0.70710678118654752440) {
    m = __dmul_rn(m, 2.0);
    e -= 1;
  }
  const double ed = static_cast<double>(e);
  const double s = __ddiv_rn(__dsub_rn(m, 1.0), __dadd_rn(m, 1.0));
  const double s2 = __dmul_rn(s, s);
  double p = 1.0 / 25.0;
#pragma unroll
  for (int k = 23; k >= 1; k -= 2) p = __dadd_rn(__dmul_rn(p, s2), 1.0 / static_cast<double>(k));
  return __dadd_rn(__dadd_rn(__dmul_rn(ed, kLn2Hi), __dmul_rn(__dmul_rn(2.0, s), p)), __dmul_rn(ed, kLn2Lo));
}

// floats <-> integers whose order is the float order (for atomicMin / atomicMax)
__device__ __forceinline__ int float_to_ordered(float f) {
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF); }
// doubles -> unsigned integers in the same order
__device__ __forceinline__ uint64_t double_to_sortable(double d) {
  const uint64_t b = static_cast<uint64_t>(__double_as_longlong(d));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// ------------------------------------------------------------------------------------------------ scenes and lines
// Where line l's points and RNG identity come from: the points of scene line_scene[l], starting at
// scene_off[line_scene[l]], and (seeds[l], line_ids[l]).  Scene indices (candidates, `indices`, the RNG counter) are
// always within the line's own scene.  One scene is the case K = 1.
struct Lines {
  const long long* scene_off;  // (K+1) first point of every scene
  const int* line_scene;       // (L)
  const uint64_t* seeds;       // (L)
  const uint32_t* line_ids;    // (L)
  int K;
  __device__ __forceinline__ bool bad(int l) const { return static_cast<unsigned>(line_scene[l]) >= static_cast<unsigned>(K); }
  __device__ __forceinline__ long long base(int l) const { return scene_off[line_scene[l]]; }
  __device__ __forceinline__ uint64_t seed_of(int l) const { return seeds[l]; }
  __device__ __forceinline__ uint64_t id_of(int l) const { return static_cast<uint64_t>(line_ids[l]); }
};

// The lines of a call grouped by scene (group_kernel): order[first[k] .. first[k+1]) are the lines of scene k, in
// no particular order (nothing downstream depends on it: per-line counters, candidates sorted before use).
struct Groups {
  const long long* scene_off;  // (K+1)
  const int* first;            // (K+1)
  const int* order;            // (L)
  int K;
};

// largest k in [lo, hi] with off[k] <= i (the scene of point i; an empty scene k has off[k] == off[k+1] and is skipped)
__device__ __forceinline__ int scene_of(const long long* __restrict__ off, int lo, int hi, long long i) {
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// One block: counting sort of the lines by scene.  Lines whose scene is out of range join no group (select_kernel flags
// them).  Global counters are read back through L2 (__ldcg) after the block's atomics.
__global__ void __launch_bounds__(1024) group_kernel(const int* __restrict__ line_scene, int L, int K, int* __restrict__ first,
                                                     int* __restrict__ cursor, int* __restrict__ order) {
  __shared__ int part[1024];
  __shared__ int carry;
  for (int k = threadIdx.x; k < K; k += blockDim.x) cursor[k] = 0;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    const int k = line_scene[l];
    if (static_cast<unsigned>(k) < static_cast<unsigned>(K)) atomicAdd(&cursor[k], 1);
  }
  __syncthreads();
  for (int b = 0; b < K; b += blockDim.x) {
    const int k = b + threadIdx.x;
    const int v = k < K ? __ldcg(cursor + k) : 0;
    part[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < blockDim.x; o <<= 1) {
      const int t = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
      __syncthreads();
      part[threadIdx.x] += t;
      __syncthreads();
    }
    if (k < K) first[k] = carry + part[threadIdx.x] - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry += part[threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.x == 0) first[K] = carry;
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) cursor[k] = __ldcg(first + k);
  __syncthreads();
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    const int k = line_scene[l];
    if (static_cast<unsigned>(k) < static_cast<unsigned>(K)) order[atomicAdd(&cursor[k], 1)] = l;
  }
}

// squared distance exactly as the oracle: (dx*dx + dy*dy) + dz*dz in double, no contraction
__device__ __forceinline__ double dist2_exact(double px, double py, double pz, const double* q) {
  const double dx = __dsub_rn(px, q[0]), dy = __dsub_rn(py, q[1]), dz = __dsub_rn(pz, q[2]);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// ------------------------------------------------------------------------------------------------ polyline resampling
// resample_polyline (src/dataset.py:8-30) for every line to 32 and to 200 points, the centroid of the 32 (src/dataset.py:
// 232) and the centred line - the same IEEE double operations in the same order as numpy (norm = sqrt((dx^2+dy^2)+dz^2),
// sequential cumsum, linspace = i * (total / (n-1)) with the last point pinned, np.interp = slope * (t - x_j) + f_j with
// the exact-hit and right-edge rules), so the results are bit-equal to the host formulation.  One block per line.
constexpr int kMaxVertices = 2048;
__global__ void __launch_bounds__(256)
resample_kernel(const double* __restrict__ verts, const long long* __restrict__ offsets, int L, double* __restrict__ line32,
                double* __restrict__ dense, double* __restrict__ centers, float* __restrict__ noisy_centered) {
  __shared__ double cum[kMaxVertices];
  __shared__ double l32[kLine * 3];
  __shared__ double ctr[3];
  const int l = blockIdx.x;
  if (l >= L) return;
  const double* v = verts + offsets[l] * 3;
  const int n = static_cast<int>(offsets[l + 1] - offsets[l]);
  if (threadIdx.x == 0 && n >= 2) {
    double c = 0.0;
    cum[0] = 0.0;
    for (int i = 1; i < n; ++i) {
      const double dx = __dsub_rn(v[3 * i], v[3 * i - 3]), dy = __dsub_rn(v[3 * i + 1], v[3 * i - 2]), dz = __dsub_rn(v[3 * i + 2], v[3 * i - 1]);
      const double seg = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
      c = i == 1 ? seg : __dadd_rn(c, seg);
      cum[i] = c;
    }
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t < kLine + kDense) {
    const int num = t < kLine ? kLine : kDense;
    const int i = t < kLine ? t : t - kLine;
    double out[3] = {0.0, 0.0, 0.0};
    if (n >= 2) {
      const double total = cum[n - 1];
      const double step = __ddiv_rn(total, static_cast<double>(num - 1));
      double x = step == 0.0 ? __dmul_rn(__ddiv_rn(static_cast<double>(i), static_cast<double>(num - 1)), total)
                             : __dmul_rn(static_cast<double>(i), step);
      if (i == num - 1) x = total;
      // j = last vertex with cum[j] <= x
      int lo = 0, hi = n - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (cum[mid] <= x) lo = mid; else hi = mid - 1;
      }
      const int j = lo;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        if (j >= n - 1) {
          out[k] = v[3 * (n - 1) + k];
        } else if (cum[j] == x) {
          out[k] = v[3 * j + k];
        } else {
          const double slope = __ddiv_rn(__dsub_rn(v[3 * j + 3 + k], v[3 * j + k]), __dsub_rn(cum[j + 1], cum[j]));
          out[k] = __dadd_rn(__dmul_rn(slope, __dsub_rn(x, cum[j])), v[3 * j + k]);
        }
      }
    }
    double* dst = t < kLine ? line32 + (static_cast<size_t>(l) * kLine + i) * 3 : dense + (static_cast<size_t>(l) * kDense + i) * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      dst[k] = out[k];
      if (t < kLine) l32[3 * i + k] = out[k];
    }
  }
  __syncthreads();
  if (t < 3) {
    double s = l32[t];
    for (int i = 1; i < kLine; ++i) s = __dadd_rn(s, l32[3 * i + t]);
    s = __ddiv_rn(s, static_cast<double>(kLine));
    ctr[t] = s;
    centers[l * 3 + t] = s;
  }
  __syncthreads();
  if (t < kLine * 3) noisy_centered[static_cast<size_t>(l) * kLine * 3 + t] = static_cast<float>(__dsub_rn(l32[t], ctr[t % 3]));
}

// ------------------------------------------------------------------------------------------------ per-line setup
// Bounding boxes (whole polyline and its kSub pieces) grown by (radius + eps), fp32 copy of the points, counters reset.
// A scene point within the radius of some polyline point lies inside that point's piece box, so testing only the
// pieces whose box contains the scene point decides `distance < radius` exactly.
__global__ void prep_kernel(const double* __restrict__ dense, int L, float grow, float* __restrict__ aabb,
                            float* __restrict__ dense_f, int* __restrict__ count, int* __restrict__ fill,
                            int* __restrict__ imin, int* __restrict__ imax) {
  const int l = blockIdx.x;
  if (l >= L) return;
  __shared__ float lo_s[kSub][3], hi_s[kSub][3];
  for (int i = threadIdx.x; i < kDense * 3; i += blockDim.x)
    dense_f[static_cast<size_t>(l) * kDense * 3 + i] = static_cast<float>(dense[static_cast<size_t>(l) * kDense * 3 + i]);
  if (threadIdx.x < kSub * 3) {
    const int sub = threadIdx.x / 3, k = threadIdx.x % 3;
    float lo = 3.4e38f, hi = -3.4e38f;
    for (int i = 0; i < kSubLen; ++i) {
      const double v = dense[(static_cast<size_t>(l) * kDense + sub * kSubLen + i) * 3 + k];
      lo = fminf(lo, __double2float_rd(v));
      hi = fmaxf(hi, __double2float_ru(v));
    }
    lo_s[sub][k] = lo;
    hi_s[sub][k] = hi;
    aabb[l * kBoxFloats + 6 * (1 + sub) + k] = lo - grow;
    aabb[l * kBoxFloats + 6 * (1 + sub) + 3 + k] = hi + grow;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int k = threadIdx.x;
    float lo = lo_s[0][k], hi = hi_s[0][k];
    for (int sub = 1; sub < kSub; ++sub) {
      lo = fminf(lo, lo_s[sub][k]);
      hi = fmaxf(hi, hi_s[sub][k]);
    }
    aabb[l * kBoxFloats + k] = lo - grow;
    aabb[l * kBoxFloats + 3 + k] = hi + grow;
  }
  if (threadIdx.x == 0) {
    count[l] = 0;
    fill[l] = 0;
    imin[l] = 0x7FFFFFFF;
    imax[l] = static_cast<int>(0x80000000u);
  }
}

// ------------------------------------------------------------------------------------------------ tube crop
// `pts` may be the scene in any order (`perm[i]` = scene index of pts[i], or null for the identity): in a spatially sorted
// order (Morton, scene.prepare_scene) the 32 points of a warp are neighbours, so a warp only enters the piece tests of
// the few lines that actually pass near it instead of diverging on most lines.
// One thread per scene point, all lines: box tests (line, then pieces), fp32 minimum distance to the points of the
// pieces whose box contains it, and the exact double evaluation only inside the band where fp32 cannot decide
// `distance < radius`.
// FILL = false: count the candidates of every line (+ intensity range).  FILL = true: write their scene indices.
// `pts` holds K scenes back to back (grp.scene_off) and a point is tested only against the lines of its own scene
// (grp.order[grp.first[k] .. grp.first[k+1])); a block whose scenes have no line in the call exits at once.  The
// candidate written is the point's index within its scene.
template <bool FILL>
__global__ void __launch_bounds__(256) tube_crop_kernel(const float4* __restrict__ pts, long long S,
                                                        const float* __restrict__ aabb, const float* __restrict__ dense_f,
                                                        const double* __restrict__ dense, double radius, float r2_lo, float r2_hi,
                                                        int* __restrict__ count, int* __restrict__ imin, int* __restrict__ imax,
                                                        int* __restrict__ fill, const long long* __restrict__ offset,
                                                        long long capacity, const int* __restrict__ perm,
                                                        uint32_t* __restrict__ cand, Groups grp) {
  __shared__ float box[kLineTile * 6];
  __shared__ int line_s[kLineTile];
  __shared__ int s_k0, s_k1;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < S) p = pts[i];
  auto inside = [&](const float* b) { return !(p.x < b[0] || p.y < b[1] || p.z < b[2] || p.x > b[3] || p.y > b[4] || p.z > b[5]); };
  if (threadIdx.x == 0) {
    const long long b0 = static_cast<long long>(blockIdx.x) * blockDim.x;
    const long long b1 = min(b0 + static_cast<long long>(blockDim.x), S) - 1;
    s_k0 = scene_of(grp.scene_off, 0, grp.K - 1, b0);
    s_k1 = scene_of(grp.scene_off, s_k0, grp.K - 1, b1);
  }
  __syncthreads();
  // grouped line positions [g_lo, g_hi) of this block's scenes, [my_lo, my_hi) of this thread's scene
  const int k0 = s_k0, k1 = s_k1;
  const int g_lo = grp.first[k0], g_hi = grp.first[k1 + 1];
  if (g_lo >= g_hi) return;  // no line of the call in this block's scenes (uniform over the block)
  const int k = (k0 == k1 || i >= S) ? k0 : scene_of(grp.scene_off, k0, k1, i);
  const int my_lo = grp.first[k], my_hi = grp.first[k + 1];
  const long long base = grp.scene_off[k];
  for (int l0 = g_lo; l0 < g_hi; l0 += kLineTile) {
    const int nl = min(kLineTile, g_hi - l0);
    __syncthreads();
    for (int t = threadIdx.x; t < nl; t += blockDim.x) line_s[t] = grp.order[l0 + t];
    __syncthreads();
    for (int t = threadIdx.x; t < nl * 6; t += blockDim.x) box[t] = aabb[line_s[t / 6] * kBoxFloats + t % 6];
    __syncthreads();
    if (i >= S) continue;
    for (int j = max(my_lo - l0, 0), j_end = min(my_hi - l0, nl); j < j_end; ++j) {
      if (!inside(box + j * 6)) continue;
      const int l = line_s[j];
      const float* sb = aabb + l * kBoxFloats + 6;
      const float* q = dense_f + static_cast<size_t>(l) * kDense * 3;
      float best = 3.4e38f;
      uint32_t pieces = 0;
      for (int sub = 0; sub < kSub; ++sub) {
        float b6[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) b6[k] = __ldg(sb + 6 * sub + k);
        if (!inside(b6)) continue;
        pieces |= 1u << sub;
        for (int k = sub * kSubLen; k < (sub + 1) * kSubLen; ++k) {
          const float dx = p.x - __ldg(q + 3 * k), dy = p.y - __ldg(q + 3 * k + 1), dz = p.z - __ldg(q + 3 * k + 2);
          best = fminf(best, dx * dx + dy * dy + dz * dz);
        }
      }
      if (best > r2_hi) continue;
      if (best >= r2_lo) {  // undecidable in fp32: the reference's float64 comparison
        const double* qd = dense + static_cast<size_t>(l) * kDense * 3;
        double bd = 1e300;
        for (int sub = 0; sub < kSub; ++sub)
          if (pieces >> sub & 1)
            for (int k = sub * kSubLen; k < (sub + 1) * kSubLen; ++k) bd = fmin(bd, dist2_exact(p.x, p.y, p.z, qd + 3 * k));
        if (!(sqrt(bd) < radius)) continue;
      }
      if (!FILL) {
        atomicAdd(&count[l], 1);
        const int o = float_to_ordered(p.w);
        atomicMin(&imin[l], o);
        atomicMax(&imax[l], o);
      } else {
        const long long pos = offset[l] + atomicAdd(&fill[l], 1);
        if (pos < capacity) cand[pos] = perm ? static_cast<uint32_t>(perm[i]) : static_cast<uint32_t>(i - base);
      }
    }
  }
}

// exclusive scan of the per-line counts (one block); status[0] = total candidates, status[1] |= 1 on overflow
__global__ void scan_kernel(const int* __restrict__ count, int L, long long capacity, long long* __restrict__ offset,
                            long long* __restrict__ status) {
  __shared__ long long carry;
  __shared__ long long part[1024];
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < L; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const long long v = i < L ? count[i] : 0;
    part[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < blockDim.x; o <<= 1) {
      const long long t = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
      __syncthreads();
      part[threadIdx.x] += t;
      __syncthreads();
    }
    if (i < L) offset[i] = carry + part[threadIdx.x] - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry += part[threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    offset[L] = carry;
    status[0] = carry;
    status[1] = carry > capacity ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------ sampling keys
// Efraimidis-Spirakis key of every candidate of the lines that have more candidates than samples:
// key = det_log(u) / w, w = det_exp(-d / decay) * (0.5 + normalised intensity)   (src/dataset.py:94-112)
__global__ void __launch_bounds__(256) sample_keys_kernel(const float4* __restrict__ pts, const double* __restrict__ line32,
                                                          const int* __restrict__ count, const long long* __restrict__ offset,
                                                          const int* __restrict__ imin, const int* __restrict__ imax, int N,
                                                          double decay, Lines src, const long long* __restrict__ status,
                                                          const uint32_t* __restrict__ cand, uint64_t* __restrict__ keys) {
  const int l = blockIdx.y;
  const int n = count[l];
  if (n <= N || status[1]) return;
  pts += src.base(l);
  const uint64_t seed = src.seed_of(l), line = src.id_of(l);
  __shared__ double lp[kLine * 3];
  for (int t = threadIdx.x; t < kLine * 3; t += blockDim.x) lp[t] = line32[static_cast<size_t>(l) * kLine * 3 + t];
  __syncthreads();
  const float lo = ordered_to_float(imin[l]), hi = ordered_to_float(imax[l]);
  const float span = __fadd_rn(__fsub_rn(hi, lo), 1e-6f);
  const long long off = offset[l];
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n; c += gridDim.x * blockDim.x) {
    const uint32_t idx = cand[off + c];
    const float4 p = pts[idx];
    double bd = 1e300;
#pragma unroll 4
    for (int k = 0; k < kLine; ++k) bd = fmin(bd, dist2_exact(p.x, p.y, p.z, lp + 3 * k));
    const double d = sqrt(bd);
    const float norm = hi > lo ? __fdiv_rn(__fsub_rn(p.w, lo), span) : 0.5f;
    const float iw = __fadd_rn(0.5f, norm);
    const double w = __dmul_rn(det_exp(__ddiv_rn(-d, decay)), static_cast<double>(iw));
    const double key = __ddiv_rn(det_log(det_uniform(seed, line, idx)), w);
    keys[off + c] = double_to_sortable(key);
  }
}

// ------------------------------------------------------------------------------------------------ selection
// key descending, then index ascending
__device__ __forceinline__ bool before(uint64_t ka, uint32_t ia, uint64_t kb, uint32_t ib) {
  return ka > kb || (ka == kb && ia < ib);
}
__device__ void bitonic_sort(uint64_t* k, uint32_t* v, int n /* power of two */) {
  for (int size = 2; size <= n; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const bool in_order = before(k[lo], v[lo], k[hi], v[hi]);
        if (in_order != up) {
          const uint64_t tk = k[lo];
          k[lo] = k[hi];
          k[hi] = tk;
          const uint32_t tv = v[lo];
          v[lo] = v[hi];
          v[hi] = tv;
        }
      }
    }
  __syncthreads();
}

// One block per line: pick the N samples and write the normalised context rows.
//   count == 0      : N zero points                                   (src/dataset.py:87-88)
//   count <= N      : uniform with replacement over the candidates     (src/dataset.py:89-91)
//   count  > N      : the N largest keys (radix select + sort)         (src/dataset.py:128, RNG contract)
__global__ void __launch_bounds__(256) select_kernel(const float4* __restrict__ pts, const double* __restrict__ centers,
                                                     const int* __restrict__ count, const long long* __restrict__ offset, int N,
                                                     int cap /* power of two >= 2 N */, Lines src,
                                                     long long* __restrict__ status, const uint32_t* __restrict__ cand,
                                                     const uint64_t* __restrict__ keys, float* __restrict__ context,
                                                     long long* __restrict__ indices, int* __restrict__ counts_out) {
  extern __shared__ uint8_t sm_raw[];
  uint64_t* sk = reinterpret_cast<uint64_t*>(sm_raw);
  uint32_t* sv = reinterpret_cast<uint32_t*>(sk + cap);
  __shared__ int hist[256];
  __shared__ uint64_t s_prefix;
  __shared__ int s_rank, s_n;
  const int l = blockIdx.x;
  const int n = count[l];
  if (threadIdx.x == 0) counts_out[l] = n;
  if (src.bad(l)) {  // scene number out of range: the line joined no group; reported, nothing written
    if (threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned long long*>(&status[1]), 4ull);
    return;
  }
  if (status[1] & 1) return;  // candidate buffer too small: the host re-runs with status[0] entries
  pts += src.base(l);
  const long long off = offset[l];
  const double cx = centers[l * 3], cy = centers[l * 3 + 1], cz = centers[l * 3 + 2];
  float* ctx = context + static_cast<size_t>(l) * N * 4;
  long long* ind = indices + static_cast<size_t>(l) * N;

  if (n <= N) {
    // candidates in ascending scene-index order
    for (int t = threadIdx.x; t < cap; t += blockDim.x) {
      sk[t] = 0;  // equal keys: the sort is by index
      sv[t] = t < n ? cand[off + t] : 0xFFFFFFFFu;
    }
    if (n > 1) bitonic_sort(sk, sv, cap); else __syncthreads();
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
      long long idx = -1;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n > 0) {
        const double u = det_uniform(src.seed_of(l), src.id_of(l), (1ull << 40) + j);
        long long pick = static_cast<long long>(__dmul_rn(u, static_cast<double>(n)));
        pick = pick < n - 1 ? pick : n - 1;
        idx = sv[pick];
        p = pts[idx];
      }
      ind[j] = idx;
      reinterpret_cast<float4*>(ctx)[j] = make_float4(static_cast<float>(__dsub_rn(p.x, cx)), static_cast<float>(__dsub_rn(p.y, cy)),
                                                      static_cast<float>(__dsub_rn(p.z, cz)), p.w);
    }
    return;
  }

  // radix select: T = N-th largest key (most significant byte first)
  if (threadIdx.x == 0) {
    s_prefix = 0;
    s_rank = N;
  }
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    for (int t = threadIdx.x; t < 256; t += blockDim.x) hist[t] = 0;
    __syncthreads();
    const uint64_t prefix = s_prefix;
    const uint64_t mask = pass == 0 ? 0 : (~0ull << (shift + 8));
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
      const uint64_t k = keys[off + c];
      if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int rank = s_rank, b = 255;
      for (; b > 0; --b) {
        if (hist[b] >= rank) break;
        rank -= hist[b];
      }
      s_rank = rank;
      s_prefix = prefix | (static_cast<uint64_t>(b) << shift);
    }
    __syncthreads();
  }
  const uint64_t T = s_prefix;
  // gather everything >= T (N entries unless several keys equal T exactly), sort, keep the first N
  if (threadIdx.x == 0) s_n = 0;
  for (int t = threadIdx.x; t < cap; t += blockDim.x) {
    sk[t] = 0;
    sv[t] = 0xFFFFFFFFu;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < n; c += blockDim.x) {
    const uint64_t k = keys[off + c];
    if (k >= T) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < cap) {
        sk[pos] = k;
        sv[pos] = cand[off + c];
      }
    }
  }
  __syncthreads();
  if (s_n > cap) {  // more than cap - N candidates share the threshold key exactly
    if (threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned long long*>(&status[1]), 2ull);
    return;
  }
  bitonic_sort(sk, sv, cap);
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const long long idx = sv[j];
    const float4 p = pts[idx];
    ind[j] = idx;
    reinterpret_cast<float4*>(ctx)[j] = make_float4(static_cast<float>(__dsub_rn(p.x, cx)), static_cast<float>(__dsub_rn(p.y, cy)),
                                                    static_cast<float>(__dsub_rn(p.z, cz)), p.w);
  }
}

}  // namespace scene
}  // namespace lrn
