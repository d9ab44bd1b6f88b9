// (a) TMA-staged pad + cyclic roll + strided window partition / reverse for the reference's channels-first layout.
//
//   x      [B][C][H][W][D]   (D contiguous)   <->   tokens [B][P][N][C]   (C contiguous)
//
// The x side is the awkward one: a window column p2 touches every P2-th W line (windows are STRIDED, reference
// swin_block.py:292-299), rolled and padded.  Viewing W as (a, r) with w = a*P2 + r turns the ww lines of one
// (sample, rolled h row, window column) tile into a dense 5-D box
//        { D: whole line, r: one residue, a: ww consecutive, h: one row, channel: a whole chunk }
// of the tensor [B*C][H][W/P2][P2][D], so ONE cp.async.bulk.tensor (TMA) instruction moves the tile, and the
// hardware's out-of-bounds handling does the zero padding on loads (negative / too large coordinates read as 0)
// and the crop on stores (out-of-bounds elements are not written).  The roll only rotates the a rows (an index
// rotation) and the D positions inside a line (a per-line offset table in shared memory).
//
// partition:  TMA load -> smem [c][a'][D_box]  --transpose-->  smem token blocks  -> coalesced 16-byte stores
// reverse  :  coalesced 16-byte loads (+ fused residual add) -> smem token blocks --transpose--> smem [c][a'][D_box]
//             -> TMA store
// Persistent CTAs, 2-4 per SM, one staged tile each: the partition kernel issues the next tile's TMA load as soon as the
// current one has left shared memory (a deeper ring of loads was measured no faster than more resident CTAs).  Pure byte
// movement: bit-exact by construction.
//
// Shared-memory layouts are chosen so that both sides of the transposition are bank-conflict free:
//   * D_box = padded line length rounded up to an ODD number of 16-byte chunks: lanes that differ in a' hit
//     different bank groups on the 16-byte side;
//   * token blocks (window p3, w' position t2) hold wd tokens x CT channels and are padded to a pitch of
//     4 (mod 32) words: lanes that differ in t2 hit different banks on the 4-byte side.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace pwa {
using namespace tc;

namespace {

// Measured on B200 (profiles/r1_tma_partition.md): one 43 KB box of 384 lines x 96(+16) bytes takes the SM's TMA unit
// ~3.4 us (~17 clk per line) whatever the pipeline depth, the split into several boxes or the number of warps (256 ->
// 1024 threads made it slower), i.e. the kernels are bound by the TMA line rate for short lines, not by the SM side.
constexpr int kPartThreads = 256;
constexpr int kRevThreads = 256;
constexpr int kWW = 8;            // lanes are mapped as (a' = lane & 7, channel word = lane >> 3)

struct TmaPartParams {
  int B, C, CT, nchunk;
  int H, W, D, Hp, Wp, Dp;
  int P1, P2, P3, P, N;
  int wd;
  int sh, sw, sd;
  int loh, low, lod;
  int dbox;          // elements per staged line
  int cw;            // channel words per token in this chunk (CT * eb / 4)
  int bp;            // token block pitch in words
  int src_bytes;     // one staged x tile, rounded up to 128 bytes
  int box_bytes;     // exact bytes one TMA box transfers
  int ntiles;
  int d0, dsh;       // TMA start coordinate along D (16-byte aligned, <= -lod) and the column shift it leaves: column j = dp + dsh
  FastDiv div_perblk, div_cpt;
};

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

struct Tile {
  int b, ah, p2, chunk;     // sample, rolled h coordinate, window column, channel chunk
  int h;                    // unpadded row of x (may be out of range: padding row / cropped row)
  int t1, p1;               // ah = t1 * P1 + p1
  int q;                    // staged row a' holds token position t2 = (a' - q) mod ww
  int r, a0;                // TMA start coordinates along the (r, a) split of W
  bool h_ok;
  __device__ __forceinline__ Tile(const TmaPartParams& p, int tile) {
    chunk = tile % p.nchunk;
    int t = tile / p.nchunk;
    p2 = t % p.P2;
    t /= p.P2;
    ah = t % p.Hp;
    b = t / p.Hp;
    t1 = ah / p.P1;
    p1 = ah - t1 * p.P1;
    h = (ah + p.sh) % p.Hp - p.loh;
    h_ok = h >= 0 && h < p.H;
    // padded-frame w of token position t2: ((t2 + q) mod ww) * P2 + rp ; unpadded w = that - low
    const int s = p2 + p.sw;
    q = s / p.P2;
    const int rp = s - q * p.P2;
    const int rr = rp - p.low;
    const int fl = rr >= 0 ? rr / p.P2 : -((-rr + p.P2 - 1) / p.P2);
    r = rr - fl * p.P2;
    a0 = fl;
  }
};

// shared-memory carve-up (dynamic smem base is 128-byte aligned)
struct Carve {
  uint8_t* src;
  uint32_t* dst;
  int* doff;
};
__device__ __forceinline__ Carve carve(uint8_t* smem, const TmaPartParams& p) {
  Carve c;
  c.src = smem;
  c.dst = reinterpret_cast<uint32_t*>(smem + p.src_bytes);
  c.doff = reinterpret_cast<int*>(c.dst + (size_t)p.P3 * kWW * p.bp);
  return c;
}

// word offset of the token block slot of staged column j (padded-frame line position dp = j - dsh): block (p3, t2 = 0),
// token t3; -1 for columns outside the padded line
__device__ __forceinline__ void fill_doff(int* doff, const TmaPartParams& p) {
  for (int j = threadIdx.x; j < p.dbox; j += blockDim.x) {
    const int dp = j - p.dsh;
    int v = -1;
    if (dp >= 0 && dp < p.Dp) {
      int dr = dp - p.sd;
      dr += dr < 0 ? p.Dp : 0;
      const int t3 = dr / p.P3, p3 = dr - t3 * p.P3;
      v = p3 * kWW * p.bp + t3 * p.cw;
    }
    doff[j] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// in-smem transposition between the staged x tile [c][a'][dbox] and the token blocks
// ---------------------------------------------------------------------------------------------
template <int EB, bool TO_TOKENS, int NT>
__device__ __forceinline__ void transpose_tile(uint8_t* src, uint32_t* dst, const int* doff, const TmaPartParams& p, int q) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ap = lane & 7, cl = lane >> 3;
  const int t2 = (ap - q + 2 * kWW) & (kWW - 1);
  constexpr int EPV = 16 / EB;                               // line positions per 16-byte vector
  const int ndv = (p.Dp + p.dsh + EPV - 1) / EPV;
  const int nch = EB == 2 ? p.cw : p.CT;                     // lanes walk channel WORDS (bf16 pairs) / channels (fp32)
  const int ncg = (nch + 3) / 4;
  const size_t cstride = (size_t)kWW * p.dbox * EB;          // bytes between channels
  for (int item = warp; item < ndv * ncg; item += NT / 32) {
    const int cg = item / ndv, dvec = item - cg * ndv;
    const int ci = cg * 4 + cl;
    if (ci >= nch) continue;
    const int4* op = reinterpret_cast<const int4*>(doff + dvec * EPV);
    uint32_t* db = dst + t2 * p.bp + ci;
    if (EB == 4) {
      uint8_t* s0 = src + (size_t)ci * cstride + ((size_t)ap * p.dbox + dvec * 4) * 4;
      const int4 o = op[0];
      const int off[4] = {o.x, o.y, o.z, o.w};
      if (TO_TOKENS) {
        const uint4 v = *reinterpret_cast<const uint4*>(s0);
        const uint32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (off[j] >= 0) db[off[j]] = vv[j];
      } else {
        uint32_t vv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) vv[j] = off[j] >= 0 ? db[off[j]] : 0u;
        *reinterpret_cast<uint4*>(s0) = make_uint4(vv[0], vv[1], vv[2], vv[3]);
      }
    } else {
      // word ci = channels (2ci, 2ci+1); 2x2 transposes between (channel, d-pair) and (d, channel-pair) words
      uint8_t* s0 = src + (size_t)(2 * ci) * cstride + ((size_t)ap * p.dbox + dvec * 8) * 2;
      const int4 o0 = op[0], o1 = op[1];
      const int off[8] = {o0.x, o0.y, o0.z, o0.w, o1.x, o1.y, o1.z, o1.w};
      if (TO_TOKENS) {
        const uint4 a = *reinterpret_cast<const uint4*>(s0);
        const uint4 b = *reinterpret_cast<const uint4*>(s0 + cstride);
        const uint32_t av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (off[2 * j] >= 0) db[off[2 * j]] = __byte_perm(av[j], bv[j], 0x5410);
          if (off[2 * j + 1] >= 0) db[off[2 * j + 1]] = __byte_perm(av[j], bv[j], 0x7632);
        }
      } else {
        uint32_t av[4], bv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t lo = off[2 * j] >= 0 ? db[off[2 * j]] : 0u;
          const uint32_t hi = off[2 * j + 1] >= 0 ? db[off[2 * j + 1]] : 0u;
          av[j] = __byte_perm(lo, hi, 0x5410);
          bv[j] = __byte_perm(lo, hi, 0x7632);
        }
        *reinterpret_cast<uint4*>(s0) = make_uint4(av[0], av[1], av[2], av[3]);
        *reinterpret_cast<uint4*>(s0 + cstride) = make_uint4(bv[0], bv[1], bv[2], bv[3]);
      }
    }
  }
}

// token-side addressing of 16-byte piece i of the tile: block = (p3, t2), token t3, piece j
struct Piece {
  uint32_t soff;      // word offset in the token-block buffer
  size_t goff;        // word offset in the token tensor
};
__device__ __forceinline__ Piece piece(const TmaPartParams& p, const Tile& t, uint32_t i) {
  uint32_t blk, rem, t3, j;
  p.div_perblk.divmod(i, blk, rem);
  p.div_cpt.divmod(rem, t3, j);
  const uint32_t p3 = blk >> 3, t2 = blk & 7;
  Piece pc;
  pc.soff = blk * p.bp + t3 * p.cw + j * 4;
  const size_t row = ((size_t)t.b * p.P + ((size_t)t.p1 * p.P2 + t.p2) * p.P3 + p3) * p.N + ((size_t)t.t1 * kWW + t2) * p.wd + t3;
  pc.goff = row * (size_t)(p.cw * p.nchunk) + (size_t)t.chunk * p.cw + j * 4;
  return pc;
}

template <int EB>
__global__ void __launch_bounds__(kPartThreads, 4) partition_tma_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                    uint32_t* __restrict__ tok, const TmaPartParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t full;
  const Carve cv = carve(smem, p);
  const int tid = threadIdx.x;
  fill_doff(cv.doff, p);
  if (tid == 0) {
    mbar_init(&full, 1);
    fence_mbar_init();
  }
  __syncthreads();
  auto issue = [&](int tile) {
    const Tile t(p, tile);
    if (!t.h_ok) return;                                   // a padding row: nothing to load, the tile is all zeros
    mbar_expect_tx(&full, (uint32_t)p.box_bytes);
    tma_load_5d(cv.src, &xmap, &full, p.d0, t.r, t.a0, t.h, t.b * p.C + t.chunk * p.CT);
  };
  if (tid == 0 && blockIdx.x < p.ntiles) issue(blockIdx.x);
  uint32_t phase = 0u;
  const uint32_t npieces = (uint32_t)p.P3 * kWW * p.div_perblk.d;
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const Tile t(p, tile);
    if (t.h_ok) {
      mbar_wait(&full, phase);
      phase ^= 1u;
      transpose_tile<EB, true, kPartThreads>(cv.src, cv.dst, cv.doff, p, t.q);
    } else {
      for (uint32_t i = tid; i < (uint32_t)p.P3 * kWW * p.bp / 4; i += kPartThreads)
        reinterpret_cast<uint4*>(cv.dst)[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();                                       // (B) token blocks complete
    for (uint32_t i = tid; i < npieces; i += kPartThreads) {
      const Piece pc = piece(p, t, i);
      *reinterpret_cast<uint4*>(tok + pc.goff) = *reinterpret_cast<const uint4*>(cv.dst + pc.soff);
    }
    __syncthreads();                                       // (C) token blocks and the staged tile are free again
    if (tid == 0 && tile + (int)gridDim.x < p.ntiles) issue(tile + gridDim.x);
  }
}

template <int EB, bool H> __device__ __forceinline__ uint32_t addw(uint32_t a, uint32_t b) {
  if (EB == 4) return __float_as_uint(__uint_as_float(a) + __uint_as_float(b));
  if (H) {                                                   // fp16 pair
    const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&a)), fb = __half22float2(*reinterpret_cast<const __half2*>(&b));
    const __half2 r = __floats2half2_rn(fa.x + fb.x, fa.y + fb.y);
    return *reinterpret_cast<const uint32_t*>(&r);
  }
  const float2 fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a));
  const float2 fb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b));
  const __nv_bfloat162 r = __floats2bfloat162_rn(fa.x + fb.x, fa.y + fb.y);
  return *reinterpret_cast<const uint32_t*>(&r);
}

template <int EB, bool ADD, bool H = false>
__global__ void __launch_bounds__(kRevThreads, 4) reverse_tma_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                  const uint32_t* __restrict__ tok,
                                                                  const uint32_t* __restrict__ tok2, const TmaPartParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const Carve cv = carve(smem, p);
  const int tid = threadIdx.x;
  fill_doff(cv.doff, p);
  __syncthreads();
  const uint32_t npieces = (uint32_t)p.P3 * kWW * p.div_perblk.d;
  constexpr int U = 3;                                     // independent 16-byte loads in flight per thread
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const Tile t(p, tile);
    if (!t.h_ok) continue;                                 // this rolled row is cropped away entirely (uniform per CTA)
    for (uint32_t i0 = tid; i0 < npieces; i0 += kRevThreads * U) {
      uint4 v[U], w[U];
      Piece pc[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t i = i0 + u * kRevThreads;
        if (i < npieces) {
          pc[u] = piece(p, t, i);
          v[u] = __ldg(reinterpret_cast<const uint4*>(tok + pc[u].goff));
          if (ADD) w[u] = __ldg(reinterpret_cast<const uint4*>(tok2 + pc[u].goff));
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t i = i0 + u * kRevThreads;
        if (i < npieces) {
          if (ADD) v[u] = make_uint4(addw<EB, H>(v[u].x, w[u].x), addw<EB, H>(v[u].y, w[u].y), addw<EB, H>(v[u].z, w[u].z), addw<EB, H>(v[u].w, w[u].w));
          *reinterpret_cast<uint4*>(cv.dst + pc[u].soff) = v[u];
        }
      }
    }
    if (tid == 0) tma_wait_read0();                        // the previous tile's TMA store has finished reading the staged tile
    __syncthreads();
    transpose_tile<EB, false, kRevThreads>(cv.src, cv.dst, cv.doff, p, t.q);
    fence_proxy_async_smem();                              // generic-proxy writes -> visible to the TMA (async proxy)
    __syncthreads();
    if (tid == 0) {
      tma_store_5d(&xmap, cv.src, p.d0, t.r, t.a0, t.h, t.b * p.C + t.chunk * p.CT);   // out-of-bounds = crop
      tma_commit();
    }
  }
  if (tid == 0) tma_wait_all0();
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}

// staged x tile + token blocks + line offset table
size_t smem_bytes(const TmaPartParams& p) {
  return (size_t)p.src_bytes + (size_t)p.P3 * kWW * p.bp * 4 + (size_t)p.dbox * 4 + 16;
}

// Measured (profiles/r1_tma_partition.md): two or more resident CTAs per SM beat one CTA with a 3-deep TMA pipeline
// (24 vs 29 us), so a tile (one staged x box + the token blocks) is sized for >= 2 CTAs per SM when the shape allows.
constexpr size_t kSmemBudget = 200 * 1024;
constexpr size_t kSmemTwoCtas = 110 * 1024;

bool plan(TmaPartParams& p, int B, int C, const pwa_geom* g, const int32_t* lo, int eb) {
  if (g->ws[1] != kWW) return false;
  p.B = B; p.C = C;
  p.H = g->dims[0]; p.W = g->dims[1]; p.D = g->dims[2];
  p.Hp = g->sp[0]; p.Wp = g->sp[1]; p.Dp = g->sp[2];
  p.P1 = g->nwin[0]; p.P2 = g->nwin[1]; p.P3 = g->nwin[2];
  p.P = g->P; p.N = g->N;
  p.wd = g->ws[2];
  p.sh = g->shift[0]; p.sw = g->shift[1]; p.sd = g->shift[2];
  p.loh = lo[0]; p.low = lo[1]; p.lod = lo[2];
  if (p.W % p.P2 != 0) return false;                              // W must split as (a, r)
  if ((p.D * eb) % 16 != 0 || (C * eb) % 16 != 0) return false;     // TMA strides / 16-byte token pieces
  const int epv = 16 / eb;
  // the innermost TMA start coordinate must be 16-byte aligned (a start of -lod with lod % epv != 0 faults): start at
  // the aligned coordinate below it and keep the shift
  const int la = (p.lod + epv - 1) / epv * epv;
  p.d0 = -la;
  p.dsh = la - p.lod;
  int chunks = (p.Dp + p.dsh + epv - 1) / epv;
  chunks |= 1;                                                     // odd number of 16-byte chunks per staged line
  p.dbox = chunks * epv;
  if (p.dbox > 256) return false;
  // channel chunk: all channels if the tile fits (double-buffered, else single), otherwise halve
  for (int pass = 0; pass < 2; ++pass)                             // pass 0: tiles that leave room for two CTAs per SM
  for (int ct = C; ct >= epv; ct /= 2) {
    if (C % ct != 0 || (ct * eb) % 16 != 0 || ct > 256) continue;
    p.CT = ct;
    p.nchunk = C / ct;
    p.cw = ct * eb / 4;
    const int blk = p.wd * p.cw;
    if (blk % 4 != 0) continue;
    p.bp = blk + ((36 - blk % 32) % 32);                           // pitch = 4 (mod 32) words, a multiple of 4
    p.box_bytes = ct * kWW * p.dbox * eb;
    p.src_bytes = (p.box_bytes + 127) & ~127;
    if (smem_bytes(p) <= (pass == 0 ? kSmemTwoCtas : kSmemBudget)) {
      const int cpt = p.cw / 4;
      if ((size_t)p.P3 * kWW * p.wd * cpt >= 65536) return false;
      p.div_perblk = FastDiv(p.wd * cpt);
      p.div_cpt = FastDiv(cpt);
      p.ntiles = B * p.Hp * p.P2 * p.nchunk;
      return true;
    }
  }
  return false;
}

bool make_map(CUtensorMap* map, const void* x, const TmaPartParams& p, int eb) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return false;
  const cuuint64_t dims[5] = {(cuuint64_t)p.D, (cuuint64_t)p.P2, (cuuint64_t)(p.W / p.P2), (cuuint64_t)p.H,
                              (cuuint64_t)p.B * p.C};
  const cuuint64_t strides[4] = {(cuuint64_t)p.D * eb, (cuuint64_t)p.P2 * p.D * eb, (cuuint64_t)p.W * p.D * eb,
                                 (cuuint64_t)p.H * p.W * p.D * eb};
  const cuuint32_t box[5] = {(cuuint32_t)p.dbox, 1u, (cuuint32_t)kWW, 1u, (cuuint32_t)p.CT};
  const cuuint32_t es[5] = {1u, 1u, 1u, 1u, 1u};
  const CUresult rc = enc(map, eb == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, const_cast<void*>(x),
                          dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS;
}

template <typename K>
bool set_smem(K kern, size_t bytes) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess;
}

}  // namespace

// Returns PWA_OK when the TMA kernel was launched, PWA_ERR_UNSUPPORTED when the shape is outside its envelope (the
// caller then uses the vector / word / generic kernels of partition.cu), another error code on failure.
int partition_tma_run(bool is_partition, const void* src, const void* src2, void* dst, int B, int C, const pwa_geom* g,
                      const int32_t* lo, int eb, bool f16, cudaStream_t st) {
  TmaPartParams p;
  // TMA stores fault on negative start coordinates (measured on B200, driver 580): padded geometries, whose crop
  // needs them, keep the vector kernel on the store side; loads zero-fill out-of-bounds boxes as documented
  if (!is_partition && g->padded) return PWA_ERR_UNSUPPORTED;
  if (!plan(p, B, C, g, lo, eb)) return PWA_ERR_UNSUPPORTED;
  const void* xptr = is_partition ? src : dst;
  if (((uintptr_t)src | (uintptr_t)src2 | (uintptr_t)dst) & 15) return PWA_ERR_UNSUPPORTED;
  CUtensorMap map;
  if (!make_map(&map, xptr, p, eb)) return PWA_ERR_UNSUPPORTED;
  const size_t smem = smem_bytes(p);
  int per_sm = (int)((227 * 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
  int grid = 148 * per_sm;
  if (grid > p.ntiles) grid = p.ntiles;
  bool ok;
  if (is_partition) {
    if (eb == 2) {
      ok = set_smem(partition_tma_kernel<2>, smem);
      if (ok) partition_tma_kernel<2><<<grid, kPartThreads, smem, st>>>(map, (uint32_t*)dst, p);
    } else {
      ok = set_smem(partition_tma_kernel<4>, smem);
      if (ok) partition_tma_kernel<4><<<grid, kPartThreads, smem, st>>>(map, (uint32_t*)dst, p);
    }
  } else {
#define PWA_REV(EBV, ...)                                                                                               \
  ok = set_smem(reverse_tma_kernel<EBV, __VA_ARGS__>, smem);                                                             \
  if (ok) reverse_tma_kernel<EBV, __VA_ARGS__><<<grid, kRevThreads, smem, st>>>(map, (const uint32_t*)src, (const uint32_t*)src2, p)
    if (eb == 2 && src2 && f16) { PWA_REV(2, true, true); }
    else if (eb == 2 && src2) { PWA_REV(2, true); }
    else if (eb == 2) { PWA_REV(2, false); }
    else if (src2) { PWA_REV(4, true); }
    else { PWA_REV(4, false); }
#undef PWA_REV
  }
  if (!ok) {
    set_error("partition_tma: cudaFuncSetAttribute(%zu bytes of shared memory) failed", smem);
    return PWA_ERR_CUDA;
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

}  // namespace pwa
