// Mesh-quality metrics: the two pytorch3d operators behind the Chamfer metric of BaseModel.validation_epoch_end
// (src/models/model_base.py:82-102).
//
//   nearest_kernel       exact brute-force nearest neighbour of every x_i in y (the per-point minima chamfer_distance reduces).
//                        y is staged through shared memory in tiles of kNnTile points, every thread holds kNnQ queries in
//                        registers and scans j in increasing order with a strict `<`, so the lowest index wins a tie.  When N
//                        alone cannot fill one wave of resident CTAs, blockIdx.y splits M into chunks; the partial minima are
//                        merged with a 64-bit atomicMin on (float bits of d) << 32 | j.  d >= 0, so its bit pattern orders like its value and the key
//                        orders by distance, then by lowest index: the merged result is the unsplit scan's, bit for bit.
//   nearest_unpack       key -> (d, j) after a split launch.
//
//   area_scan_kernel     face areas 1/2 |(v1-v0) x (v2-v0)| in fp64 and the inclusive prefix sum (CDF) of the areas, fp64,
//   area_scan_blocks     in three levels that are each a SEQUENTIAL running sum: kScanItems faces per thread, the threads of a
//   area_scan_add        block by one thread, the blocks by one thread.  Every CDF entry is prefix + local running sum with the
//                        prefix of a group equal to the rounded end of the previous group, so the CDF is non-decreasing and a
//                        zero-area face repeats its predecessor's value exactly (a parallel tree scan guarantees neither).
//   sample_kernel        one thread per sample: a 53-bit uniform r picks the first face with cdf[i] > r * total (binary search:
//                        a zero-area face is never chosen), two 24-bit uniforms give the barycentric weights
//                        w0 = 1 - sqrt(u), w1 = sqrt(u) (1 - v), w2 = sqrt(u) v (pytorch3d's _rand_barycentric_coords).
//
// Compiled with -fmad=false; the pair distance is written with explicit round-to-nearest intrinsics anyway, so
// d = ((dx*dx) + (dy*dy)) + (dz*dz) with every operation rounded in fp32 whatever the flag.
#include <cfloat>
#include <math_constants.h>

#include "nm_common.h"
#include "nm_composite.cuh"

namespace nm {
namespace {

constexpr int kNnThreads = 256;
constexpr int kNnQ = 4;                         // queries per thread
constexpr int kNnBlockQ = kNnThreads * kNnQ;    // queries per CTA
constexpr int kNnTile = 512;                    // y points per shared-memory tile (8 KB)

__device__ __forceinline__ float pair_d2(float ax, float ay, float az, float4 b) {
  const float dx = __fsub_rn(ax, b.x), dy = __fsub_rn(ay, b.y), dz = __fsub_rn(az, b.z);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// CTA (bx, by): queries [bx*kNnBlockQ, +kNnBlockQ) against y[by*chunk, min(M, (by+1)*chunk)).  keys == nullptr: one chunk
// covers all of y, the result is written directly.
__global__ void __launch_bounds__(kNnThreads) nearest_kernel(const float* __restrict__ x, long long N, const float* __restrict__ y,
                                                             long long M, long long chunk, float* __restrict__ d_out,
                                                             int* __restrict__ j_out, unsigned long long* __restrict__ keys) {
  __shared__ float4 s_y[kNnTile];
  const long long m0 = (long long)blockIdx.y * chunk;
  const long long m1 = (m0 + chunk < M) ? m0 + chunk : M;
  const long long i0 = (long long)blockIdx.x * kNnBlockQ + threadIdx.x;
  float qx[kNnQ], qy[kNnQ], qz[kNnQ], best[kNnQ];
  int bj[kNnQ];
#pragma unroll
  for (int q = 0; q < kNnQ; ++q) {
    const long long i = i0 + (long long)q * kNnThreads;
    qx[q] = qy[q] = qz[q] = 0.f;
    if (i < N) { qx[q] = x[3 * i]; qy[q] = x[3 * i + 1]; qz[q] = x[3 * i + 2]; }
    // +inf with the chunk's first index: if every distance overflows to +inf, the strict `<` never fires and the lowest
    // index still stands, as in an argmin
    best[q] = CUDART_INF_F;
    bj[q] = (int)m0;
  }
  for (long long t0 = m0; t0 < m1; t0 += kNnTile) {
    __syncthreads();
    for (int k = threadIdx.x; k < kNnTile; k += kNnThreads) {
      const long long j = t0 + k;
      // padding is NaN: every comparison with it is false, so it can never win
      s_y[k] = j < m1 ? make_float4(y[3 * j], y[3 * j + 1], y[3 * j + 2], 0.f)
                      : make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, 0.f);
    }
    __syncthreads();
    const int jb = (int)t0;
#pragma unroll 4
    for (int k = 0; k < kNnTile; ++k) {
      const float4 b = s_y[k];
#pragma unroll
      for (int q = 0; q < kNnQ; ++q) {
        const float d = pair_d2(qx[q], qy[q], qz[q], b);
        if (d < best[q]) { best[q] = d; bj[q] = jb + k; }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < kNnQ; ++q) {
    const long long i = i0 + (long long)q * kNnThreads;
    if (i >= N) continue;
    if (keys) {
      atomicMin(keys + i, ((unsigned long long)__float_as_uint(best[q]) << 32) | (unsigned)bj[q]);
    } else {
      d_out[i] = best[q];
      j_out[i] = bj[q];
    }
  }
}

__global__ void nearest_unpack(const unsigned long long* __restrict__ keys, long long N, float* __restrict__ d_out,
                               int* __restrict__ j_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const unsigned long long k = keys[i];
  d_out[i] = __uint_as_float((unsigned)(k >> 32));
  j_out[i] = (int)(unsigned)(k & 0xffffffffull);
}

// ------------------------------------------------------------------------------------------------ surface sampling
constexpr int kScanThreads = 256;
constexpr int kScanItems = 32;                                   // consecutive faces per thread
constexpr int kScanBlockFaces = kScanThreads * kScanItems;

struct FaceVerts { double a[3], b[3], c[3]; };

__device__ __forceinline__ FaceVerts load_face(const float* __restrict__ verts, const int* __restrict__ faces, long long f) {
  FaceVerts fv;
  const int i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    fv.a[k] = (double)verts[3 * (long long)i0 + k];
    fv.b[k] = (double)verts[3 * (long long)i1 + k];
    fv.c[k] = (double)verts[3 * (long long)i2 + k];
  }
  return fv;
}

__device__ __forceinline__ void face_cross(const FaceVerts& fv, double n[3]) {
  const double e1[3] = {fv.b[0] - fv.a[0], fv.b[1] - fv.a[1], fv.b[2] - fv.a[2]};
  const double e2[3] = {fv.c[0] - fv.a[0], fv.c[1] - fv.a[1], fv.c[2] - fv.a[2]};
  n[0] = e1[1] * e2[2] - e1[2] * e2[1];
  n[1] = e1[2] * e2[0] - e1[0] * e2[2];
  n[2] = e1[0] * e2[1] - e1[1] * e2[0];
}

// level 1 + 2: cdf[i] = (threads' sequential prefix) + (the thread's own running sum); blk[b] = the block's total
__global__ void __launch_bounds__(kScanThreads) area_scan_kernel(const float* __restrict__ verts, const int* __restrict__ faces,
                                                                 long long F, double* __restrict__ cdf, double* __restrict__ blk) {
  __shared__ double s_tot[kScanThreads];
  const long long f0 = (long long)blockIdx.x * kScanBlockFaces + (long long)threadIdx.x * kScanItems;
  double run = 0.0;
  for (int k = 0; k < kScanItems; ++k) {
    const long long f = f0 + k;
    if (f >= F) break;
    double n[3];
    face_cross(load_face(verts, faces, f), n);
    run = run + 0.5 * sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    cdf[f] = run;
  }
  s_tot[threadIdx.x] = run;
  __syncthreads();
  if (threadIdx.x == 0) {
    double p = 0.0;
    for (int t = 0; t < kScanThreads; ++t) { const double s = s_tot[t]; s_tot[t] = p; p = p + s; }
    blk[blockIdx.x] = p;
  }
  __syncthreads();
  const double pre = s_tot[threadIdx.x];
  for (int k = 0; k < kScanItems; ++k) {
    const long long f = f0 + k;
    if (f >= F) break;
    cdf[f] = pre + cdf[f];
  }
}

// level 3: exclusive running sum of the block totals in place; blk[nblk] = the total area
__global__ void area_scan_blocks(double* __restrict__ blk, long long nblk) {
  if (threadIdx.x != 0) return;
  double p = 0.0;
  for (long long b = 0; b < nblk; ++b) { const double s = blk[b]; blk[b] = p; p = p + s; }
  blk[nblk] = p;
}

__global__ void area_scan_add(double* __restrict__ cdf, long long F, const double* __restrict__ blk) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const long long b = f / kScanBlockFaces;
  if (b > 0) cdf[f] = blk[b] + cdf[f];
}

__global__ void sample_kernel(const float* __restrict__ verts, const int* __restrict__ faces, long long F,
                              const double* __restrict__ cdf, long long n, uint64_t seed, float* __restrict__ points,
                              int* __restrict__ face_idx, float* __restrict__ normals) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const double total = cdf[F - 1];
  if (!(total > 0.0)) {                        // no surface: zeros (pytorch3d leaves invalid meshes' samples at zero)
    points[3 * s] = points[3 * s + 1] = points[3 * s + 2] = 0.f;
    if (face_idx) face_idx[s] = -1;
    if (normals) normals[3 * s] = normals[3 * s + 1] = normals[3 * s + 2] = 0.f;
    return;
  }
  double t = u01_53(seed, 3 * (uint64_t)s) * total;
  if (!(t < total)) t = nextafter(total, 0.0);  // r * total rounded up to total: take the last face that adds area
  long long lo = 0, hi = F - 1;                 // first i with cdf[i] > t; cdf[F-1] = total > t
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (cdf[mid] > t) hi = mid;
    else lo = mid + 1;
  }
  const double u = (double)u01(seed, 3 * (uint64_t)s + 1), v = (double)u01(seed, 3 * (uint64_t)s + 2);
  const double su = sqrt(u);
  const double w0 = 1.0 - su, w1 = su * (1.0 - v), w2 = su * v;
  const FaceVerts fv = load_face(verts, faces, lo);
#pragma unroll
  for (int k = 0; k < 3; ++k) points[3 * s + k] = (float)(w0 * fv.a[k] + w1 * fv.b[k] + w2 * fv.c[k]);
  if (face_idx) face_idx[s] = (int)lo;
  if (normals) {
    double nr[3];
    face_cross(fv, nr);
    const double len = fmax(sqrt(nr[0] * nr[0] + nr[1] * nr[1] + nr[2] * nr[2]), DBL_EPSILON);
#pragma unroll
    for (int k = 0; k < 3; ++k) normals[3 * s + k] = (float)(nr[k] / len);
  }
}

struct NnPlan { long long qblocks, splits, chunk; };

// resident CTAs of nearest_kernel per SM (registers bound it: 46 x 256 threads -> 5 on sm_100a)
int nearest_ctas_per_sm() {
  static const int v = [] {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, nearest_kernel, kNnThreads, 0) != cudaSuccess || n < 1) n = 1;
    return n;
  }();
  return v;
}

NnPlan nearest_plan(long long N, long long M, int num_sms) {
  NnPlan p;
  p.qblocks = (N + kNnBlockQ - 1) / kNnBlockQ;
  const long long tiles = (M + kNnTile - 1) / kNnTile;
  const long long want = (long long)num_sms * nearest_ctas_per_sm();     // one full wave of resident CTAs
  long long splits = p.qblocks >= want ? 1 : (want + p.qblocks - 1) / p.qblocks;
  if (splits > tiles) splits = tiles;
  if (splits > 65535) splits = 65535;
  if (splits < 1) splits = 1;
  const long long tiles_per = (tiles + splits - 1) / splits;
  p.chunk = tiles_per * kNnTile;
  p.splits = (M + p.chunk - 1) / p.chunk;
  return p;
}

}  // namespace

size_t nearest_ws_bytes(long long N, long long M, int num_sms) {
  if (N <= 0 || M <= 0) return 0;
  return nearest_plan(N, M, num_sms).splits > 1 ? (size_t)N * 8 : 0;
}

int launch_nearest(const float* x, long long N, const float* y, long long M, float* d, int* j, void* ws, int num_sms,
                   cudaStream_t st, int64_t* launches) {
  if (N == 0) return 0;
  const NnPlan p = nearest_plan(N, M, num_sms);
  NM_CHECK(p.qblocks < (1ll << 31), "nearest: too many query points");
  unsigned long long* keys = nullptr;
  if (p.splits > 1) {
    keys = reinterpret_cast<unsigned long long*>(ws);
    NM_CUDA(cudaMemsetAsync(keys, 0xff, (size_t)N * 8, st));
  }
  nearest_kernel<<<dim3((unsigned)p.qblocks, (unsigned)p.splits), kNnThreads, 0, st>>>(x, N, y, M, p.chunk, d, j, keys);
  NM_CUDA(cudaGetLastError());
  if (launches) *launches += 1;
  if (keys) {
    nearest_unpack<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(keys, N, d, j);
    NM_CUDA(cudaGetLastError());
    if (launches) *launches += 1;
  }
  return 0;
}

size_t mesh_sample_ws_bytes(long long F) {
  const long long nblk = (F + kScanBlockFaces - 1) / kScanBlockFaces;
  return ((size_t)F * 8 + 255) / 256 * 256 + (size_t)(nblk + 1) * 8;
}

int launch_mesh_sample(const float* verts, const int* faces, long long F, long long n, uint64_t seed, float* points, int* face_idx,
                       float* normals, void* ws, cudaStream_t st, int64_t* launches) {
  if (n == 0) return 0;
  if (F == 0) {
    NM_CUDA(cudaMemsetAsync(points, 0, (size_t)n * 12, st));
    if (normals) NM_CUDA(cudaMemsetAsync(normals, 0, (size_t)n * 12, st));
    if (face_idx) NM_CUDA(cudaMemsetAsync(face_idx, 0xff, (size_t)n * 4, st));
    return 0;
  }
  const long long nblk = (F + kScanBlockFaces - 1) / kScanBlockFaces;
  NM_CHECK(nblk < (1ll << 31), "mesh sample: too many faces");
  double* cdf = reinterpret_cast<double*>(ws);
  double* blk = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + ((size_t)F * 8 + 255) / 256 * 256);
  area_scan_kernel<<<(unsigned)nblk, kScanThreads, 0, st>>>(verts, faces, F, cdf, blk);
  NM_CUDA(cudaGetLastError());
  area_scan_blocks<<<1, 32, 0, st>>>(blk, nblk);
  NM_CUDA(cudaGetLastError());
  area_scan_add<<<(unsigned)((F + 255) / 256), 256, 0, st>>>(cdf, F, blk);
  NM_CUDA(cudaGetLastError());
  sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(verts, faces, F, cdf, n, seed, points, face_idx, normals);
  NM_CUDA(cudaGetLastError());
  if (launches) *launches += 4;
  return 0;
}

}  // namespace nm
