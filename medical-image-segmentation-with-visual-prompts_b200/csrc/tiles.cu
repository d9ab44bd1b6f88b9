// Whole-volume sliding-window inference: patch gather, overlap-weighted stitching and the final normalise / argmax / count
// pass (include/pwa.h, "whole-volume sliding-window inference").
//
// The reference scores the downstream model on whole CT volumes by unfolding the volume into roi-sized patches, running the
// model on sub-batches of them and adding the predictions back (SegmentationTrainer.test, SURVEY.md §3(4)).  Here the patch
// origins are an int32 [n_total][4] table (b, x0, y0, z0) on the device, and every call reads its range [first, first + count)
// of that table from a device cursor {first, count}: one captured CUDA graph (gather -> predictor -> stitch -> advance) then
// walks the whole table by replaying, with no host scalar frozen into it.
//
// Stitching uses no float atomics: the voxels a call's patches cover are each owned by one thread (the one at the voxel's
// position in the first patch of the call that covers it), which reads the accumulator once, adds the terms of every covering
// patch of the call in patch order and writes it once.  Every voxel's sum is therefore formed in the global patch order, whatever
// the sub-batch size, and the result is bitwise reproducible.
#include "common.cuh"

namespace pwa {

namespace {

constexpr int kThreads = 256;
constexpr int kMaxCountClasses = 1024;          // shared-memory TP/FP/FN counters of the count pass

struct TileArgs {
  int B, C;                // C: input channels (gather) or classes (stitch)
  int X, Y, Z;
  int r0, r1, r2;
  int sw;
  long n_total;
};

// {first, count} of this call, clamped so that no read leaves the origin table or the sub-batch
__device__ __forceinline__ void read_cursor(const int32_t* cursor, const TileArgs& a, long& first, int& count) {
  first = cursor[0];
  long c = cursor[1];
  if (first < 0 || first > a.n_total) first = a.n_total;
  if (c > a.sw) c = a.sw;
  if (c > a.n_total - first) c = a.n_total - first;
  count = c < 0 ? 0 : (int)c;
}

// patches [sw][C][r0][r1][r2] (To) <- image [B][C][X][Y][Z] (Ti); one thread per V consecutive z of a patch row.
template <typename Ti, typename To, int V>
__global__ void __launch_bounds__(kThreads) tile_gather_kernel(const Ti* __restrict__ img, const int4* __restrict__ origins,
                                                               const int32_t* __restrict__ cursor, To* __restrict__ out,
                                                               TileArgs a, float cval) {
  long first;
  int count;
  read_cursor(cursor, a, first, count);
  const float cv = to_f32(from_f32<Ti>(cval));    // F.pad fills in the input's dtype, .to() then casts
  const int rv = a.r2 / V;
  const long per_patch = (long)a.C * a.r0 * a.r1 * rv;
  const long total = per_patch * a.sw;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int s = (int)(t / per_patch);
    long rem = t - (long)s * per_patch;
    const int kc = (int)(rem % rv);
    rem /= rv;
    const int j = (int)(rem % a.r1);
    rem /= a.r1;
    const int i = (int)(rem % a.r0);
    const int c = (int)(rem / a.r0);
    float v[V];
#pragma unroll
    for (int e = 0; e < V; ++e) v[e] = cv;
    if (s < count) {
      const int4 o = origins[first + s];
      const int x = o.y + i, y = o.z + j, z = o.w + kc * V;
      if (x < a.X && y < a.Y) {
        const Ti* row = img + ((((long)o.x * a.C + c) * a.X + x) * a.Y + y) * a.Z;
        if (V > 1 && z + V <= a.Z && ((uintptr_t)(row + z) & 15) == 0) {
          alignas(16) Ti t_in[V];
#pragma unroll
          for (int q = 0; q < (int)(V * sizeof(Ti) / 16); ++q)
            reinterpret_cast<uint4*>(t_in)[q] = __ldg(reinterpret_cast<const uint4*>(row + z) + q);
#pragma unroll
          for (int e = 0; e < V; ++e) v[e] = to_f32(t_in[e]);
        } else {
#pragma unroll
          for (int e = 0; e < V; ++e)
            if (z + e < a.Z) v[e] = to_f32(row[z + e]);
        }
      }
    }
    alignas(16) To t_out[V];
#pragma unroll
    for (int e = 0; e < V; ++e) t_out[e] = from_f32<To>(v[e]);
    To* dst = out + t * V;
    if constexpr (V * sizeof(To) % 16 == 0) {
#pragma unroll
      for (int q = 0; q < (int)(V * sizeof(To) / 16); ++q) reinterpret_cast<uint4*>(dst)[q] = reinterpret_cast<const uint4*>(t_out)[q];
    } else {
#pragma unroll
      for (int e = 0; e < V; ++e) dst[e] = t_out[e];
    }
  }
}

__device__ __forceinline__ bool covers(const int4& o, int b, int x, int y, int z, const TileArgs& a) {
  return o.x == b && x >= o.y && x < o.y + a.r0 && y >= o.z && y < o.z + a.r1 && z >= o.w && z < o.w + a.r2;
}

// acc [B][K][X][Y][Z] += w * pred, wsum [B][X][Y][Z] += w over the call's patches; pred [sw][K][r0][r1][r2] (Tp), w [r0][r1][r2].
template <typename Tp>
__global__ void __launch_bounds__(kThreads) tile_stitch_kernel(const Tp* __restrict__ pred, const float* __restrict__ w,
                                                               const int4* __restrict__ origins, const int32_t* __restrict__ cursor,
                                                               float* __restrict__ acc, float* __restrict__ wsum, TileArgs a) {
  extern __shared__ int4 org_s[];                 // [sw] origins of this call
  long first;
  int count;
  read_cursor(cursor, a, first, count);
  for (int s = threadIdx.x; s < count; s += blockDim.x) org_s[s] = origins[first + s];
  __syncthreads();
  const int rv = a.r0 * a.r1 * a.r2;
  const long nvox = (long)a.X * a.Y * a.Z;
  const long total = (long)count * rv;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int s = (int)(t / rv);
    const int p = (int)(t - (long)s * rv);
    const int k = p % a.r2, j = (p / a.r2) % a.r1, i = p / (a.r2 * a.r1);
    const int4 o = org_s[s];
    const int b = o.x, x = o.y + i, y = o.z + j, z = o.w + k;
    if (x >= a.X || y >= a.Y || z >= a.Z) continue;              // past the volume (an axis shorter than the roi)
    bool owner = true;
    for (int q = 0; q < s; ++q)
      if (covers(org_s[q], b, x, y, z, a)) { owner = false; break; }
    if (!owner) continue;
    const long vox = ((long)x * a.Y + y) * a.Z + z;
    float ws = wsum[(long)b * nvox + vox];
    for (int q = s; q < count; ++q) {
      const int4 oq = org_s[q];
      if (!covers(oq, b, x, y, z, a)) continue;
      ws = __fadd_rn(ws, __ldg(w + ((x - oq.y) * a.r1 + (y - oq.z)) * a.r2 + (z - oq.w)));
    }
    wsum[(long)b * nvox + vox] = ws;
    for (int c = 0; c < a.C; ++c) {
      float* dst = acc + ((long)b * a.C + c) * nvox + vox;
      float v = *dst;
      for (int q = s; q < count; ++q) {
        const int4 oq = org_s[q];
        if (!covers(oq, b, x, y, z, a)) continue;
        const int pq = ((x - oq.y) * a.r1 + (y - oq.z)) * a.r2 + (z - oq.w);
        v = __fmaf_rn(__ldg(w + pq), to_f32(pred[((long)q * a.C + c) * rv + pq]), v);
      }
      *dst = v;
    }
  }
}

__global__ void tile_advance_kernel(int32_t* cursor, int sw, long n_total) {
  const long first = (long)cursor[0] + cursor[1];
  const long left = n_total - first;
  cursor[0] = (int32_t)first;
  cursor[1] = (int32_t)(left < sw ? (left < 0 ? 0 : left) : sw);
}

template <typename T> __device__ __forceinline__ long load_label(const void* p, long i) { return (long)static_cast<const T*>(p)[i]; }

__device__ __forceinline__ long load_label_dt(const void* p, int dt, long i) {
  return dt == PWA_LABEL_U8 ? load_label<uint8_t>(p, i) : dt == PWA_LABEL_I32 ? load_label<int32_t>(p, i) : load_label<int64_t>(p, i);
}

// per-(class) TP / FP / FN of one voxel into the CTA's shared counters; voxels with a label or target outside [0, K) are skipped
__device__ __forceinline__ void count_voxel(unsigned long long* cnt, int K, long lab, long tgt) {
  if (tgt < 0 || tgt >= K || lab < 0 || lab >= K) return;
  if (lab == tgt) {
    atomicAdd(&cnt[lab], 1ull);
  } else {
    atomicAdd(&cnt[K + lab], 1ull);
    atomicAdd(&cnt[2 * K + tgt], 1ull);
  }
}

__device__ __forceinline__ void flush_counts(unsigned long long* cnt, int K, int b, int64_t* tp, int64_t* fp, int64_t* fn) {
  __syncthreads();
  for (int c = threadIdx.x; c < 3 * K; c += blockDim.x) {
    const unsigned long long v = cnt[c];
    if (v == 0) continue;
    int64_t* dst = c < K ? tp : c < 2 * K ? fp : fn;
    atomicAdd(reinterpret_cast<unsigned long long*>(dst + (long)b * K + c % K), v);
  }
}

__device__ __forceinline__ void zero_counts(unsigned long long* cnt, int K) {
  for (int c = threadIdx.x; c < 3 * K; c += blockDim.x) cnt[c] = 0ull;
  __syncthreads();
}

// one pass over acc [B][K][nvox], wsum [B][nvox]: out = acc / wsum (out_dt), labels = argmax_k (label_dt), counts vs target.
// blockIdx.y = sample, so that a CTA's counters belong to one sample.
__global__ void __launch_bounds__(kThreads) tile_finalize_kernel(const float* __restrict__ acc, const float* __restrict__ wsum,
                                                                 int K, long nvox, void* out, int out_dt, void* labels,
                                                                 int label_dt, const void* target, int target_dt, int64_t* tp,
                                                                 int64_t* fp, int64_t* fn) {
  extern __shared__ unsigned long long cnt[];     // [3][K] when counting
  const int b = blockIdx.y;
  if (target) zero_counts(cnt, K);
  for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < nvox; v += (long)gridDim.x * blockDim.x) {
    const float ws = wsum[(long)b * nvox + v];
    int best = 0;
    float bv = 0.f;
    for (int c = 0; c < K; ++c) {
      const long idx = ((long)b * K + c) * nvox + v;
      const float y = acc[idx] / ws;
      if (out) {
        if (out_dt == PWA_F32) static_cast<float*>(out)[idx] = y;
        else if (out_dt == PWA_BF16) static_cast<__nv_bfloat16*>(out)[idx] = from_f32<__nv_bfloat16>(y);
        else static_cast<__half*>(out)[idx] = from_f32<__half>(y);
      }
      // torch.argmax: the first maximum, NaN counts as the largest value
      if (c == 0 || (y > bv && !(bv != bv)) || (y != y && !(bv != bv))) {
        best = c;
        bv = y;
      }
    }
    const long li = (long)b * nvox + v;
    if (labels) {
      if (label_dt == PWA_LABEL_U8) static_cast<uint8_t*>(labels)[li] = (uint8_t)best;
      else static_cast<int32_t*>(labels)[li] = best;
    }
    if (target) count_voxel(cnt, K, best, load_label_dt(target, target_dt, li));
  }
  if (target) flush_counts(cnt, K, b, tp, fp, fn);
}

__global__ void __launch_bounds__(kThreads) seg_counts_kernel(const void* labels, int label_dt, const void* target, int target_dt,
                                                              int K, long nvox, int64_t* tp, int64_t* fp, int64_t* fn) {
  extern __shared__ unsigned long long cnt[];
  const int b = blockIdx.y;
  zero_counts(cnt, K);
  for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < nvox; v += (long)gridDim.x * blockDim.x) {
    const long li = (long)b * nvox + v;
    count_voxel(cnt, K, load_label_dt(labels, label_dt, li), load_label_dt(target, target_dt, li));
  }
  flush_counts(cnt, K, b, tp, fp, fn);
}

unsigned grid_for(long work, int per_sm) {
  long g = (work + kThreads - 1) / kThreads;
  const long cap = 148L * per_sm;
  if (g > cap) g = cap;
  return (unsigned)(g < 1 ? 1 : g);
}

bool float_dt(int dt) { return dt == PWA_F32 || dt == PWA_BF16 || dt == PWA_F16; }
bool label_dt_ok(int dt) { return dt == PWA_LABEL_U8 || dt == PWA_LABEL_I32 || dt == PWA_LABEL_I64; }

int check_tiling(const char* who, int B, int C, const int32_t dims[3], const int32_t roi[3], int sw, int64_t n_total,
                 const void* origins, const void* cursor) {
  PWA_CHECK_ARG(dims != nullptr && roi != nullptr, "%s: null dims / roi", who);
  PWA_CHECK_ARG(origins != nullptr && cursor != nullptr, "%s: null origins / cursor", who);
  PWA_CHECK_ARG(B > 0 && C > 0, "%s: B=%d C=%d", who, B, C);
  for (int a = 0; a < 3; ++a) {
    PWA_CHECK_ARG(dims[a] > 0 && roi[a] > 0, "%s: dims / roi must be positive (axis %d: %d, %d)", who, a, dims[a], roi[a]);
  }
  PWA_CHECK_ARG((int64_t)roi[0] * roi[1] * roi[2] <= (1LL << 30), "%s: roi of %d x %d x %d voxels is too large", who, roi[0],
                roi[1], roi[2]);
  PWA_CHECK_ARG(sw > 0 && sw <= PWA_TILE_MAX_SW, "%s: sw=%d (1 .. %d)", who, sw, PWA_TILE_MAX_SW);
  PWA_CHECK_ARG(n_total >= 0 && n_total < (1LL << 31), "%s: n_total=%lld", who, (long long)n_total);
  PWA_CHECK_ARG(((uintptr_t)origins & 15) == 0, "%s: origins must be 16-byte aligned", who);
  return PWA_OK;
}

TileArgs tile_args(int B, int C, const int32_t dims[3], const int32_t roi[3], int sw, int64_t n_total) {
  TileArgs a;
  a.B = B; a.C = C;
  a.X = dims[0]; a.Y = dims[1]; a.Z = dims[2];
  a.r0 = roi[0]; a.r1 = roi[1]; a.r2 = roi[2];
  a.sw = sw;
  a.n_total = n_total;
  return a;
}

template <typename Ti, typename To>
void launch_gather(const void* image, const int32_t* origins, const int32_t* cursor, void* patches, const TileArgs& a, float cval,
                   bool vec, cudaStream_t st) {
  const long work = (long)a.sw * a.C * a.r0 * a.r1 * a.r2 / (vec ? 8 : 1);
  if (vec)
    tile_gather_kernel<Ti, To, 8><<<grid_for(work, 16), kThreads, 0, st>>>((const Ti*)image, (const int4*)origins, cursor,
                                                                          (To*)patches, a, cval);
  else
    tile_gather_kernel<Ti, To, 1><<<grid_for(work, 16), kThreads, 0, st>>>((const Ti*)image, (const int4*)origins, cursor,
                                                                          (To*)patches, a, cval);
}

template <typename Ti>
void launch_gather_in(const void* image, const int32_t* origins, const int32_t* cursor, void* patches, int dtype_out,
                      const TileArgs& a, float cval, bool vec, cudaStream_t st) {
  if (dtype_out == PWA_F32) launch_gather<Ti, float>(image, origins, cursor, patches, a, cval, vec, st);
  else if (dtype_out == PWA_BF16) launch_gather<Ti, __nv_bfloat16>(image, origins, cursor, patches, a, cval, vec, st);
  else launch_gather<Ti, __half>(image, origins, cursor, patches, a, cval, vec, st);
}

}  // namespace

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_tile_gather(const void* image, int dtype_in, int B, int Cin, const int32_t dims[3], const int32_t* origins,
                               int64_t n_total, const int32_t* cursor, const int32_t roi[3], int sw, float cval, void* patches,
                               int dtype_out, void* stream) {
  int rc = check_tiling("pwa_tile_gather", B, Cin, dims, roi, sw, n_total, origins, cursor);
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(image != nullptr && patches != nullptr, "pwa_tile_gather: null image / patches");
  PWA_CHECK_ARG(float_dt(dtype_in) && float_dt(dtype_out), "pwa_tile_gather: bad dtype (in %d, out %d)", dtype_in, dtype_out);
  const TileArgs a = tile_args(B, Cin, dims, roi, sw, n_total);
  const bool vec = roi[2] % 8 == 0 && ((uintptr_t)patches & 15) == 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype_in == PWA_F32) launch_gather_in<float>(image, origins, cursor, patches, dtype_out, a, cval, vec, st);
  else if (dtype_in == PWA_BF16) launch_gather_in<__nv_bfloat16>(image, origins, cursor, patches, dtype_out, a, cval, vec, st);
  else launch_gather_in<__half>(image, origins, cursor, patches, dtype_out, a, cval, vec, st);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

extern "C" int pwa_tile_stitch(const void* pred, int dtype_pred, const float* weight, int B, int K, const int32_t dims[3],
                               const int32_t* origins, int64_t n_total, const int32_t* cursor, const int32_t roi[3], int sw,
                               float* acc, float* wsum, void* stream) {
  int rc = check_tiling("pwa_tile_stitch", B, K, dims, roi, sw, n_total, origins, cursor);
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(pred != nullptr && weight != nullptr && acc != nullptr && wsum != nullptr,
                "pwa_tile_stitch: null pred / weight / acc / wsum");
  PWA_CHECK_ARG(float_dt(dtype_pred), "pwa_tile_stitch: bad dtype %d", dtype_pred);
  const TileArgs a = tile_args(B, K, dims, roi, sw, n_total);
  const long work = (long)sw * roi[0] * roi[1] * roi[2];
  const unsigned grid = grid_for(work, 16);
  const size_t smem = (size_t)sw * sizeof(int4);
  cudaStream_t st = (cudaStream_t)stream;
  const int4* org = (const int4*)origins;
  if (dtype_pred == PWA_F32)
    tile_stitch_kernel<float><<<grid, kThreads, smem, st>>>((const float*)pred, weight, org, cursor, acc, wsum, a);
  else if (dtype_pred == PWA_BF16)
    tile_stitch_kernel<__nv_bfloat16><<<grid, kThreads, smem, st>>>((const __nv_bfloat16*)pred, weight, org, cursor, acc, wsum, a);
  else
    tile_stitch_kernel<__half><<<grid, kThreads, smem, st>>>((const __half*)pred, weight, org, cursor, acc, wsum, a);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

extern "C" int pwa_tile_advance(int32_t* cursor, int sw, int64_t n_total, void* stream) {
  PWA_CHECK_ARG(cursor != nullptr, "pwa_tile_advance: null cursor");
  PWA_CHECK_ARG(sw > 0 && sw <= PWA_TILE_MAX_SW, "pwa_tile_advance: sw=%d (1 .. %d)", sw, PWA_TILE_MAX_SW);
  PWA_CHECK_ARG(n_total >= 0 && n_total < (1LL << 31), "pwa_tile_advance: n_total=%lld", (long long)n_total);
  tile_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(cursor, sw, (long)n_total);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

static int check_counts(const char* who, int K, const void* target, int target_dt, const int64_t* tp, const int64_t* fp,
                        const int64_t* fn) {
  PWA_CHECK_ARG(target == nullptr || label_dt_ok(target_dt), "%s: bad target dtype %d", who, target_dt);
  PWA_CHECK_ARG(target == nullptr || (tp != nullptr && fp != nullptr && fn != nullptr), "%s: counting needs tp, fp and fn", who);
  PWA_CHECK_ARG(target == nullptr || K <= kMaxCountClasses, "%s: counts support at most %d classes, got %d", who, kMaxCountClasses, K);
  return PWA_OK;
}

static int zero_counts_async(int B, int K, int64_t* tp, int64_t* fp, int64_t* fn, cudaStream_t st) {
  const size_t n = (size_t)B * K * sizeof(int64_t);
  PWA_CUDA_OK(cudaMemsetAsync(tp, 0, n, st));
  PWA_CUDA_OK(cudaMemsetAsync(fp, 0, n, st));
  PWA_CUDA_OK(cudaMemsetAsync(fn, 0, n, st));
  return PWA_OK;
}

extern "C" int pwa_tile_finalize(const float* acc, const float* wsum, int B, int K, const int32_t dims[3], void* out, int dtype_out,
                                 void* labels, const void* target, int target_dtype, int64_t* tp, int64_t* fp, int64_t* fn,
                                 void* stream) {
  PWA_CHECK_ARG(acc != nullptr && wsum != nullptr && dims != nullptr, "pwa_tile_finalize: null acc / wsum / dims");
  PWA_CHECK_ARG(B > 0 && K > 0 && dims[0] > 0 && dims[1] > 0 && dims[2] > 0, "pwa_tile_finalize: B=%d K=%d dims %d x %d x %d", B, K,
                dims[0], dims[1], dims[2]);
  PWA_CHECK_ARG(B <= 65535, "pwa_tile_finalize: B=%d (at most 65535)", B);
  PWA_CHECK_ARG(out == nullptr || float_dt(dtype_out), "pwa_tile_finalize: bad output dtype %d", dtype_out);
  int rc = check_counts("pwa_tile_finalize", K, target, target_dtype, tp, fp, fn);
  if (rc != PWA_OK) return rc;
  const long nvox = (long)dims[0] * dims[1] * dims[2];
  cudaStream_t st = (cudaStream_t)stream;
  if (target) {
    rc = zero_counts_async(B, K, tp, fp, fn, st);
    if (rc != PWA_OK) return rc;
  }
  const dim3 grid(grid_for(nvox, 8), B);
  const size_t smem = target ? (size_t)3 * K * sizeof(unsigned long long) : 0;
  tile_finalize_kernel<<<grid, kThreads, smem, st>>>(acc, wsum, K, nvox, out, dtype_out, labels,
                                                     K <= 256 ? PWA_LABEL_U8 : PWA_LABEL_I32, target, target_dtype, tp, fp, fn);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

extern "C" int pwa_seg_counts(const void* labels, int label_dtype, const void* target, int target_dtype, int B, int64_t nvox, int K,
                              int64_t* tp, int64_t* fp, int64_t* fn, void* stream) {
  PWA_CHECK_ARG(labels != nullptr && target != nullptr, "pwa_seg_counts: null labels / target");
  PWA_CHECK_ARG(label_dt_ok(label_dtype), "pwa_seg_counts: bad label dtype %d", label_dtype);
  PWA_CHECK_ARG(B > 0 && B <= 65535 && nvox >= 0 && K > 0, "pwa_seg_counts: B=%d nvox=%lld K=%d", B, (long long)nvox, K);
  int rc = check_counts("pwa_seg_counts", K, target, target_dtype, tp, fp, fn);
  if (rc != PWA_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  rc = zero_counts_async(B, K, tp, fp, fn, st);
  if (rc != PWA_OK) return rc;
  if (nvox == 0) return PWA_OK;
  const dim3 grid(grid_for(nvox, 8), B);
  seg_counts_kernel<<<grid, kThreads, (size_t)3 * K * sizeof(unsigned long long), st>>>(labels, label_dtype, target, target_dtype, K,
                                                                                       (long)nvox, tp, fp, fn);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}
