// 5x5 box stencil:  out = (sum of the 25 neighbours) / 25, per channel, integer division.
// Reference: the relative_access / box_nbh2d user kernels of benchmarks/box_5x5_filter2.cc:71-81
// (image2d<int>) and examples/box_filter.cc:23-32 (image2d<vuchar3>, vint3 accumulator).
//
// Byte images (u8, vuchar3) run as byte streams: a vuchar3 row is 3*ncols bytes and the
// horizontal taps sit CS = 3 bytes apart.  Tiles are staged in shared memory by TMA
// (cp.async.bulk.tensor.2d + mbarrier); see k_box5_bytes_tma below for the two-phase scheme.
#include "common.cuh"

#include <algorithm>
#include <atomic>
#include "tma.cuh"

namespace vppb {

// ------------------------------------------------------------------ tensor map encoding
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_tensor_map_2d(CUtensorMap* map, void* origin, CUtensorMapDataType elem, int elem_bytes, uint64_t width,
                         uint64_t height, uint64_t pitch, uint32_t box_w, uint32_t box_h) {
  static std::atomic<PFN_tmapEncodeTiled> cached{nullptr};
  PFN_tmapEncodeTiled fn = cached.load(std::memory_order_acquire);
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
      set_error("cuTensorMapEncodeTiled entry point unavailable (%d)", (int)e);
      return VPPB_E_CUDA;
    }
    fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
    cached.store(fn, std::memory_order_release);
  }
  (void)elem_bytes;
  cuuint64_t gdim[2] = {width, height};
  cuuint64_t gstr[1] = {pitch};
  cuuint32_t box[2] = {box_w, box_h};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, elem, 2, origin, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): origin %p w %llu h %llu pitch %llu box %ux%u", (int)r, origin,
              (unsigned long long)width, (unsigned long long)height, (unsigned long long)pitch, box_w, box_h);
    return VPPB_E_CUDA;
  }
  return VPPB_OK;
}

// ------------------------------------------------------------------ direct kernels (any layout)
// One thread per output element; used for images the TMA path cannot describe (unaligned
// external buffers) and as the int32 path.  T = element, CS = tap stride in elements.
template <typename T, typename ACC, int CS>
__global__ void k_box5_direct(Img in, Img out, int row_elems) {
  long long total = (long long)out.nrows * row_elems;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int r = (int)(i / row_elems);
    int x = (int)(i - (long long)r * row_elems);
    ACC s = 0;
#pragma unroll
    for (int dy = -2; dy <= 2; dy++) {
      const T* p = row_ptr<T>(in, r + dy) + x;
#pragma unroll
      for (int dx = -2; dx <= 2; dx++) s += (ACC)p[dx * CS];
    }
    row_ptr<T>(out, r)[x] = (T)(s / 25);
  }
}

// ------------------------------------------------------------------ TMA tile kernel (bytes)
// One CTA per tile of 992 x 16 output bytes.  Thread 0 issues ONE TMA load of the 1024-byte x
// 20-row input box (16 bytes of halo-and-alignment left and right, 2 rows above/below) and the
// whole CTA waits on its mbarrier.
//   phase 1 (vertical): thread = (16-byte column group, 8 output rows).  Bytes are split into
//     packed 16-bit lanes E = (b0,b2), O = (b1,b3) of each word and the 5-row column sums are kept
//     as a running window in registers (ring of 5 rows), written to shared memory as u16 pairs.
//   phase 2 (horizontal + divide): thread = (row, 16-byte output group).  The 5 taps CS bytes
//     apart are whole or word-straddling lane pairs of the column sums (one PRMT each), summed
//     with IADD3, divided by 25 with an exact multiply-shift and packed back to bytes.
// 4 CTAs (16 warps) are resident per SM; every input byte is fetched once per tile (+25 % halo
// rows, served by L2).  HBM-bound: 2 bytes of traffic per output byte.
constexpr int BX_BOXW = 1024;           // bytes per box row (64 column groups of 16 bytes)
constexpr int BX_OUTW = 992;            // output bytes per tile row (62 groups)
constexpr int BX_THREADS = 128;
constexpr int BX_CS_ROW_WORDS = BX_BOXW / 4;              // 256 words per plane per row
// TH = output rows per tile (16: 4 CTAs/SM, +25 % halo rows; 8: 8 CTAs/SM, +50 % halo rows)
template <int TH> struct BoxCfg {
  static constexpr int INH = TH + 4;                          // input rows per tile
  static constexpr int RAW_BYTES = INH * BX_BOXW;
  static constexpr int CS_BYTES = TH * 2 * BX_CS_ROW_WORDS * 4;  // E and O planes
  static constexpr int SMEM = RAW_BYTES + CS_BYTES + 16;
};
constexpr unsigned BX_DIV25 = 671089u;  // floor(s/25) == (s * 671089) >> 24 for 0 <= s <= 6375 (checked exhaustively)

// a + b (and a - b) on the FMA pipe: with a runtime multiplier ptxas must keep the IMAD, which moves the
// packed-lane additions off the half-rate ALU pipe (PRMT/LOP3/IADD3/SHF) that bounds this kernel.
__device__ __forceinline__ uint32_t fadd_u32(uint32_t a, uint32_t mul, uint32_t b) { return a * mul + b; }  // mul = +1 / -1 at run time

// floor(lane / 25) of both 16-bit lanes of se (lanes x, x+2) and so (lanes x+1, x+3), packed to 4 bytes.
// lo lanes: (v * 671089) >> 24.  hi lanes: mulhi(se, 671089) = (hi*M + ((lo*M) >> 16)) >> 16, whose byte 1 is
// floor(hi/25): the carry-in (< 2^16) is far below the slack of the magic number (exhaustively checked in
// tests/test_abi.py::test_box_division_magic).
__device__ __forceinline__ uint32_t box_div_pack(uint32_t se, uint32_t so) {
  const uint32_t pel = (se & 0xFFFFu) * BX_DIV25, pol = (so & 0xFFFFu) * BX_DIV25;
  const uint32_t peh = __umulhi(se, BX_DIV25), poh = __umulhi(so, BX_DIV25);
  const uint32_t lo = __byte_perm(pel, pol, 0x0073);  // (q(x), q(x+1)): byte 3 of the products
  const uint32_t hi = __byte_perm(peh, poh, 0x0051);  // (q(x+2), q(x+3)): byte 1 of the high products
  return __byte_perm(lo, hi, 0x5410);
}

// ---------------- phase 1 of a tile: 5-row column sums of the raw box -> E / O planes in shared memory
template <int BX_TH>
__device__ __forceinline__ void box_phase1(const unsigned char* raw, uint32_t* csE, uint32_t* csO, int tid, uint32_t minus_one) {
  constexpr int RG_ROWS = BX_TH / 2;  // output rows per phase-1 row group
  const int cg = tid & 63, rg = tid >> 6;
  const unsigned char* col = raw + (rg * RG_ROWS) * BX_BOXW + cg * 16;
  uint32_t ringE[5][4], ringO[5][4], VE[4], VO[4];
#pragma unroll
  for (int q = 0; q < 4; q++) { VE[q] = 0; VO[q] = 0; }
#pragma unroll
  for (int j = 0; j < RG_ROWS + 4; j++) {
    const uint4 v = *reinterpret_cast<const uint4*>(col + j * BX_BOXW);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    const int slot = j % 5;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const uint32_t e = w[q] & 0x00FF00FFu, o = __byte_perm(w[q], 0u, 0x4341);
      if (j >= 5) {
        VE[q] = fadd_u32(ringE[slot][q], minus_one, VE[q] + e);   // V += e - old  (one IADD3 + one IMAD)
        VO[q] = fadd_u32(ringO[slot][q], minus_one, VO[q] + o);
      } else { VE[q] += e; VO[q] += o; }
      ringE[slot][q] = e;
      ringO[slot][q] = o;
    }
    if (j >= 4) {
      const int orow = rg * RG_ROWS + j - 4;
      *reinterpret_cast<uint4*>(csE + orow * BX_CS_ROW_WORDS + cg * 4) = make_uint4(VE[0], VE[1], VE[2], VE[3]);
      *reinterpret_cast<uint4*>(csO + orow * BX_CS_ROW_WORDS + cg * 4) = make_uint4(VO[0], VO[1], VO[2], VO[3]);
    }
  }
}

// ---------------- phase 2 of a tile: horizontal taps, divide, store (out_base / out_pitch: the image the tile belongs to)
template <int CS, int BX_TH>
__device__ __forceinline__ void box_phase2(const uint32_t* csE, const uint32_t* csO, unsigned char* out_base, long long out_pitch, int out_nrows,
                                           int rowbytes, int x0, int y0, int vec_store, int tid, uint32_t one) {
  const int rows_here = min(BX_TH, out_nrows - y0);
  for (int u = tid; u < BX_TH * 62; u += BX_THREADS) {
    const int row = u / 62, og = u - row * 62;
    const int x = x0 + og * 16;
    if (row >= rows_here || x >= rowbytes) continue;
    // own words are box words 4og+4 .. 4og+7 (the box starts 16 bytes left of x0); window = words k-2 .. k+5
    const uint32_t* pe = csE + row * BX_CS_ROW_WORDS + og * 4 + 2;
    const uint32_t* po = csO + row * BX_CS_ROW_WORDS + og * 4 + 2;
    const uint2 e0 = *reinterpret_cast<const uint2*>(pe), e2 = *reinterpret_cast<const uint2*>(pe + 6);
    const uint4 e1 = *reinterpret_cast<const uint4*>(pe + 2);
    const uint2 o0 = *reinterpret_cast<const uint2*>(po), o2 = *reinterpret_cast<const uint2*>(po + 6);
    const uint4 o1 = *reinterpret_cast<const uint4*>(po + 2);
    const uint32_t E[8] = {e0.x, e0.y, e1.x, e1.y, e1.z, e1.w, e2.x, e2.y};
    const uint32_t O[8] = {o0.x, o0.y, o1.x, o1.y, o1.z, o1.w, o2.x, o2.y};
    uint32_t SE[7], SO[7];
#pragma unroll
    for (int i = 0; i < 7; i++) {
      SE[i] = __byte_perm(E[i], E[i + 1], 0x5432);  // lanes (byte2 of word i, byte0 of word i+1)
      SO[i] = __byte_perm(O[i], O[i + 1], 0x5432);  // lanes (byte3 of word i, byte1 of word i+1)
    }
    uint32_t ow[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int i = j + 2;
      uint32_t he, ho;
      if (CS == 3) {
        // lanes (x, x+2): taps x-6, x-3, x, x+3, x+6 ; lanes (x+1, x+3) likewise.  3 terms on the ALU (IADD3), 2 on the FMA pipe.
        he = fadd_u32(SE[i + 1], one, fadd_u32(SO[i], one, SE[i - 2] + O[i - 1] + E[i]));
        ho = fadd_u32(SO[i + 1], one, fadd_u32(E[i + 1], one, SO[i - 2] + SE[i - 1] + O[i]));
      } else {
        he = fadd_u32(SE[i], one, fadd_u32(O[i], one, SE[i - 1] + SO[i - 1] + E[i]));  // CS == 1: taps x-2 .. x+2
        ho = fadd_u32(SO[i], one, fadd_u32(SE[i], one, SO[i - 1] + E[i] + O[i]));
      }
      ow[j] = box_div_pack(he, ho);
    }
    unsigned char* dst = out_base + (long long)(y0 + row) * out_pitch + x;
    if (vec_store && x + 16 <= rowbytes) {
      *reinterpret_cast<uint4*>(dst) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    } else {
      for (int k = 0; k < 16; k++)
        if (x + k < rowbytes) dst[k] = (unsigned char)(ow[k >> 2] >> ((k & 3) * 8));
    }
  }
}

// Persistent: each CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...; the TMA load of the NEXT tile is
// issued right after phase 1 (the raw box is dead once the column sums are in shared memory), so its
// latency hides behind phase 2.
template <int CS, int BX_TH>
__global__ void __launch_bounds__(BX_THREADS, BX_TH == 16 ? 4 : 6) k_box5_bytes_tma(const __grid_constant__ CUtensorMap tmap, Img out, int rowbytes, int strips,
                                                                 int ntiles, int vec_store, uint32_t one) {
  constexpr int BX_RAW_BYTES = BoxCfg<BX_TH>::RAW_BYTES, BX_CS_BYTES = BoxCfg<BX_TH>::CS_BYTES;
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* raw = smem;
  uint32_t* csE = reinterpret_cast<uint32_t*>(smem + BX_RAW_BYTES);
  uint32_t* csO = csE + BX_TH * BX_CS_ROW_WORDS;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + BX_RAW_BYTES + BX_CS_BYTES);
  const int tid = threadIdx.x;
  const uint32_t minus_one = 0u - one;
  grid_launch_dependents();
  if (tid == 0) mbar_init(bar, 1);
  grid_dependency_wait();  // launched programmatically behind the previous kernel of the stream

  if (tid == 0) {
    fence_barrier_init();
    mbar_arrive_expect_tx(bar, BX_RAW_BYTES);
    // tensor origin = 16 bytes left of x = 0, 2 rows above y = 0; elements are 8 bytes; the box starts at
    // x0 - 16.  (Measured on B200: the innermost box coordinate times the element size must be a multiple
    // of 16 bytes, otherwise UTMALDG raises "illegal instruction" - dbg/tma_test.cu.)
    tma_load_2d(raw, &tmap, (blockIdx.x % strips) * (BX_OUTW / 8), (blockIdx.x / strips) * BX_TH, bar);
  }
  __syncthreads();  // barrier init visible to the waiters
  uint32_t parity = 0;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int x0 = (tile % strips) * BX_OUTW, y0 = (tile / strips) * BX_TH;
    mbar_wait(bar, parity);
    parity ^= 1;
    box_phase1<BX_TH>(raw, csE, csO, tid, minus_one);
    __syncthreads();
    // the raw box is dead: prefetch the next tile of this CTA behind phase 2
    if (tid == 0 && tile + (int)gridDim.x < ntiles) {
      const int nt = tile + gridDim.x;
      mbar_arrive_expect_tx(bar, BX_RAW_BYTES);
      tma_load_2d(raw, &tmap, (nt % strips) * (BX_OUTW / 8), (nt / strips) * BX_TH, bar);
    }
    box_phase2<CS, BX_TH>(csE, csO, out.base, out.pitch, out.nrows, rowbytes, x0, y0, vec_store, tid, one);
    __syncthreads();  // column sums consumed before the next tile's phase 1 overwrites them
  }
}

// The same walk over the tiles of a BATCH of equally shaped images in ONE launch (a video batch: the frames of a step):
// global tile g = image * tiles_per_image + tile, every image has its own tensor map and output base.  The ramp-up and
// tail of a launch (a few microseconds, comparable to a whole 1080p frame) are paid once per batch instead of once per
// frame, and the prefetch chain never drains between frames.  The maps live in the kernel parameter space
// (__grid_constant__): TMA reads them in place.
constexpr int BX_MAX_BATCH = 32;
struct BoxBatch {
  CUtensorMap maps[BX_MAX_BATCH];
  unsigned char* out_base[BX_MAX_BATCH];
};

template <int CS, int BX_TH>
__global__ void __launch_bounds__(BX_THREADS, BX_TH == 16 ? 4 : 6) k_box5_bytes_tma_batch(const __grid_constant__ BoxBatch batch, int nimg, int out_pitch, int out_nrows,
                                                                       int rowbytes, int strips, int tiles_per_image, int vec_store, uint32_t one) {
  constexpr int BX_RAW_BYTES = BoxCfg<BX_TH>::RAW_BYTES, BX_CS_BYTES = BoxCfg<BX_TH>::CS_BYTES;
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* raw = smem;
  uint32_t* csE = reinterpret_cast<uint32_t*>(smem + BX_RAW_BYTES);
  uint32_t* csO = csE + BX_TH * BX_CS_ROW_WORDS;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + BX_RAW_BYTES + BX_CS_BYTES);
  const int tid = threadIdx.x;
  const uint32_t minus_one = 0u - one;
  const int total = nimg * tiles_per_image;

  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
    if ((int)blockIdx.x < total) {
      const int img = blockIdx.x / tiles_per_image, tile = blockIdx.x - img * tiles_per_image;
      mbar_arrive_expect_tx(bar, BX_RAW_BYTES);
      tma_load_2d(raw, &batch.maps[img], (tile % strips) * (BX_OUTW / 8), (tile / strips) * BX_TH, bar);
    }
  }
  __syncthreads();  // barrier init visible to the waiters
  uint32_t parity = 0;

  for (int g = blockIdx.x; g < total; g += gridDim.x) {
    const int img = g / tiles_per_image, tile = g - img * tiles_per_image;
    const int x0 = (tile % strips) * BX_OUTW, y0 = (tile / strips) * BX_TH;
    mbar_wait(bar, parity);
    parity ^= 1;
    box_phase1<BX_TH>(raw, csE, csO, tid, minus_one);
    __syncthreads();
    if (tid == 0 && g + (int)gridDim.x < total) {  // prefetch this CTA's next tile (possibly of the next image) behind phase 2
      const int ng = g + gridDim.x;
      const int nimg_ = ng / tiles_per_image, nt = ng - nimg_ * tiles_per_image;
      mbar_arrive_expect_tx(bar, BX_RAW_BYTES);
      tma_load_2d(raw, &batch.maps[nimg_], (nt % strips) * (BX_OUTW / 8), (nt / strips) * BX_TH, bar);
    }
    box_phase2<CS, BX_TH>(csE, csO, batch.out_base[img], out_pitch, out_nrows, rowbytes, x0, y0, vec_store, tid, one);
    __syncthreads();  // column sums consumed before the next tile's phase 1 overwrites them
  }
}

// ------------------------------------------------------------------ streaming kernel (bytes)
// The work is cut into UNITS: 128 output bytes of the rows of one row chunk (R rows of one image).  A WARP takes BS_UPW = 4
// consecutive units in the flattened (image, row chunk, column unit) order - they may lie in different row chunks or images -
// so a row whose byte width is a multiple of 128 leaves no lane without work.  8 lanes share a unit, each owning BS_LW = 4
// output words, and the warp walks its units down their chunks in lockstep.  Per stage of BS_K = 5 input rows, lanes 0..3
// each fetch their unit's 160 x 5 byte TMA box (16 bytes left + 128 + 16 right) into a ring of BS_STAGES stages; the stage
// mbarrier takes one arrival per unit.  No CTA-wide barrier anywhere, and the pipeline keeps running from one task of the
// warp into its next one.  Per input row a lane
//   loads its window from the stage (LDS.64 + LDS.128 + LDS.64: bytes x-8 .. x+23),
//   splits the words into packed 16-bit lanes O = (b1,b3) (one PRMT) and E = (b0,b2) = w - 256 O (one IMAD),
//   forms the 5 horizontal taps CS bytes apart (whole or word-straddling lane pairs, one PRMT each) -> H, 8 registers,
//   slides the vertical window in registers: S += H - H(5 rows ago) (a ring of 5 rows, statically indexed because a stage
//     is exactly 5 rows),
//   and for every completed window divides by 25 (exact multiply-shift) and stores its 16 bytes.
// Horizontal-first means the only data exchanged between lanes is the raw halo, which TMA already put in shared memory:
// no shared-memory writes, no __syncthreads; one __syncwarp per stage before its buffer is handed back to TMA.
// The ALU pipe (PRMT / IADD3 / LOP3) and the FMA pipe (IMAD) each take a warp instruction every other cycle.  The byte split
// and the divide use IMADs with run-time multipliers (-256, 2^16), which ptxas cannot turn back into ALU instructions; the
// additions are left to ptxas, which moves some of them to the FMA pipe as IMAD.IADD.  A steady-state row then issues about
// as many instructions as twice either pipe's share (profiles/r3_box_stream.md).
// A task is R = 5 m - 4 output rows, exactly m stages.  A stage after the first whose 5 rows all lie inside every unit's
// chunk, in a warp whose lanes all store whole 16-byte words, runs without any per-row predicate.  The first stage of a task
// (input rows 0..3 complete no window), a stage past the last row of an image and a warp with lanes at the right edge of the
// image take the checked path.
constexpr int BS_K = 5;            // rows per stage == rows of the vertical window
constexpr int BS_MAX_BATCH = 128;  // images per launch of the streaming kernel (their tensor maps travel in the 32 KB kernel parameter space)
constexpr int BS_LW = 4;                                              // output words per lane
constexpr int BS_UNIT = 128;                                          // output bytes of a unit row
constexpr int BS_LPU = BS_UNIT / (4 * BS_LW);                         // lanes per unit (8)
constexpr int BS_UPW = 32 / BS_LPU;                                   // units per warp (4)
constexpr int BS_BOXW = BS_UNIT + 32;                                 // bytes per box row (160)
constexpr int BS_UNIT_BYTES = ((BS_K * BS_BOXW + 127) / 128) * 128;   // one unit's box in a stage (TMA destinations are 128-byte aligned)
constexpr int BS_STAGE_BYTES = BS_UPW * BS_UNIT_BYTES;
constexpr int BS_WARPS = 4;
constexpr int BS_STAGES = 3;
constexpr int BS_CTAS_PER_SM = 4;  // 16 warps per SM: at most 128 registers per thread
constexpr int BS_SMEM = BS_WARPS * BS_STAGES * (BS_STAGE_BYTES + 8);

template <int NB>
struct BoxStream {
  CUtensorMap maps[NB];
  unsigned char* out_base[NB];
  // row tiles (multi-GPU): pixel (0,0) of the tile itself and of the tiles above / below it (NULL: none, the tile's own
  // border rows are the halo).  The neighbours' memory may be a peer GPU's, mapped into this process.
  const unsigned char* in_base[NB];
  const unsigned char* up_base[NB];
  const unsigned char* dn_base[NB];
  int out_pitch, nrows, rowbytes, ucols, chunks, R, groups, vec_store, units, tasks;
  int in_pitch, row_room;   // row_room: addressable bytes of a row from pixel (0,0) to the end of its pitch
  uint32_t one;
};

// floor(lane / 25) of the four 16-bit lanes of (se, so) packed to bytes (q(x), q(x+1), q(x+2), q(x+3)); all four
// multiplies are high products (lo lanes moved up by a multiply by 2^16 on the FMA pipe), quotients in byte 1.
__device__ __forceinline__ uint32_t box_div_pack_hi(uint32_t se, uint32_t so, uint32_t shl16) {
  const uint32_t pel = __umulhi(se * shl16, BX_DIV25), pol = __umulhi(so * shl16, BX_DIV25);
  const uint32_t peh = __umulhi(se, BX_DIV25), poh = __umulhi(so, BX_DIV25);
  const uint32_t lo = __byte_perm(pel, pol, 0x0051);
  const uint32_t hi = __byte_perm(peh, poh, 0x0051);
  return __byte_perm(lo, hi, 0x5410);
}

// the partial store of a lane that straddles the right edge of the image, or of an unaligned output (kept out of the hot loop)
__device__ __noinline__ void box_store_partial(unsigned char* d, const uint32_t* ow, int nbytes) {
  for (int k = 0; k < nbytes; k++) d[k] = (unsigned char)(ow[k >> 2] >> ((k & 3) * 8));
}

// One input row of a lane: rp = its window in the stage (8 bytes left of its first output byte).  Leaves the horizontal
// 5-sums of the row in (rE, rO) (the ring slot of this row, which held the row 5 rows up) and slides (SE, SO) by them.
template <int CS>
__device__ __forceinline__ void box_stream_row(const unsigned char* rp, uint32_t (&rE)[BS_LW], uint32_t (&rO)[BS_LW], uint32_t (&SE)[BS_LW],
                                               uint32_t (&SO)[BS_LW], uint32_t m256) {
  constexpr int NW = BS_LW + 4;  // words of a lane's window: 2 left + BS_LW own + 2 right
  static_assert(BS_LW == 4, "the window is loaded as 2 + 4 + 2 words");
  const uint2 wl = *reinterpret_cast<const uint2*>(rp);
  const uint4 wm = *reinterpret_cast<const uint4*>(rp + 8);
  const uint2 wr = *reinterpret_cast<const uint2*>(rp + 24);
  const uint32_t w[NW] = {wl.x, wl.y, wm.x, wm.y, wm.z, wm.w, wr.x, wr.y};
  uint32_t E[NW], O[NW], XE[NW - 1], XO[NW - 1];
#pragma unroll
  for (int i = 0; i < NW; i++) {
    O[i] = __byte_perm(w[i], 0u, 0x4341);  // (b1, b3)
    E[i] = fadd_u32(O[i], m256, w[i]);     // (b0, b2) = w - 256 O, on the FMA pipe
  }
#pragma unroll
  for (int i = 0; i < NW - 1; i++) { XE[i] = __byte_perm(E[i], E[i + 1], 0x5432); XO[i] = __byte_perm(O[i], O[i + 1], 0x5432); }
#pragma unroll
  for (int q = 0; q < BS_LW; q++) {
    const int i = q + 2;
    uint32_t he, ho;
    if (CS == 3) {  // lanes (x, x+2): taps x-6, x-3, x, x+3, x+6; lanes (x+1, x+3) likewise
      he = XE[i + 1] + XO[i] + XE[i - 2] + O[i - 1] + E[i];
      ho = XO[i + 1] + E[i + 1] + XO[i - 2] + XE[i - 1] + O[i];
    } else {        // CS == 1: taps x-2 .. x+2
      he = XE[i] + O[i] + XE[i - 1] + XO[i - 1] + E[i];
      ho = XO[i] + XE[i] + XO[i - 1] + E[i] + O[i];
    }
    SE[q] = SE[q] + he - rE[q];  // one IADD3 with a negated operand
    SO[q] = SO[q] + ho - rO[q];
    rE[q] = he;
    rO[q] = ho;
  }
}

// A stage that straddles a row-tile seam, for one unit: row by row, each from the tile that owns it - the halo rows come
// straight from the neighbour's (peer GPU's) memory as 1-D bulk copies, so the transfer is part of the kernel's own load pipeline.
template <int NB>
__device__ __noinline__ void box_stage_from_tiles(const BoxStream<NB>& p, unsigned char* dst, uint64_t* bar, int img, int ucol, int ty) {
  const unsigned char* up = p.up_base[img];
  const unsigned char* dn = p.dn_base[img];
  const int xoff = ucol * BS_UNIT - 16;
  const int len = min(BS_BOXW, p.row_room - xoff);
  int rows = 0;
  for (int i = 0; i < BS_K; i++) rows += (ty + i - 2 <= p.nrows + 1) ? 1 : 0;
  mbar_arrive_expect_tx(bar, rows * len);
  for (int i = 0; i < BS_K; i++) {
    const int v = ty + i - 2;  // image row of the tile
    if (v > p.nrows + 1) continue;
    const unsigned char* src = (v < 0 && up) ? up + (long long)(p.nrows + v) * p.in_pitch
                             : (v >= p.nrows && dn) ? dn + (long long)(v - p.nrows) * p.in_pitch
                                                    : p.in_base[img] + (long long)v * p.in_pitch;
    tma_load_1d(dst + i * BS_BOXW, src + xoff, len, bar);
  }
}

template <int CS, int NB>
__global__ void __launch_bounds__(BS_WARPS * 32, BS_CTAS_PER_SM) k_box5_stream(const __grid_constant__ BoxStream<NB> p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* ring = smem + warp * (BS_STAGES * BS_STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BS_WARPS * BS_STAGES * BS_STAGE_BYTES) + warp * BS_STAGES;
  const int gw = blockIdx.x * BS_WARPS + warp, nw = gridDim.x * BS_WARPS;
  const int per_img = p.chunks * p.ucols;
  const uint32_t m256 = 0u - (p.one << 8), shl16 = p.one << 16;  // -256 and 2^16, unknown to ptxas: the multiplies stay IMADs

  grid_launch_dependents();  // the next kernel of the stream may be scheduled while this one drains (it waits before it reads)
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < BS_STAGES; s++) mbar_init(&bars[s], BS_UPW);  // one arrival per unit
    fence_barrier_init();
  }
  __syncwarp();
  grid_dependency_wait();    // launched programmatically: everything above overlapped the previous kernel's tail; its writes are visible now

  // producer cursor of lanes 0 .. BS_UPW - 1 (lane = the unit of the warp's task it fetches): the next stage is rows
  // [py, py + 5) of tensor map pimg at unit column pcol; pleft stages remain in the current task (the same in every lane).
  // A task is decoded once (two divisions); only stages that straddle a row-tile seam take the (out-of-line) row-by-row path.
  int ptask = gw - nw, pslot = 0, pimg = 0, pcol = 0, py = 0, pleft = 0;
  bool pvalid = false, pseam = false;
  auto produce = [&]() {
    if (pleft == 0) {
      ptask += nw;
      if (ptask < p.tasks) {
        const int u = ptask * BS_UPW + lane;
        pvalid = u < p.units;  // the last task of a launch may hold fewer units
        int chunk = 0;
        if (pvalid) {
          pimg = u / per_img;
          const int rem = u - pimg * per_img;
          chunk = rem / p.ucols;
          pcol = rem - chunk * p.ucols;
        }
        py = chunk * p.R;
        pleft = p.groups;
        pseam = pvalid && ((p.up_base[pimg] && py < 2) || (p.dn_base[pimg] && py + p.groups * BS_K > p.nrows + 2));
      }
    }
    if (pleft > 0) {
      unsigned char* dst = ring + pslot * BS_STAGE_BYTES + lane * BS_UNIT_BYTES;
      if (!pvalid)
        mbar_arrive(&bars[pslot]);
      else if (pseam && ((p.up_base[pimg] && py < 2) || (p.dn_base[pimg] && py + BS_K > p.nrows + 2)))
        box_stage_from_tiles<NB>(p, dst, &bars[pslot], pimg, pcol, py);
      else {
        mbar_arrive_expect_tx(&bars[pslot], BS_K * BS_BOXW);
        // tensor origin = 16 bytes left of x = 0 and 2 rows above y = 0; 8-byte elements (x coordinate * 8 is a multiple of 16)
        tma_load_2d(dst, &p.maps[pimg], pcol * (BS_UNIT / 8), py, &bars[pslot]);
      }
      py += BS_K;
      pleft--;
    }
    pslot = (pslot + 1 == BS_STAGES) ? 0 : pslot + 1;
  };
  if (lane < BS_UPW) {
#pragma unroll 1
    for (int s = 0; s < BS_STAGES; s++) produce();
  }

  const int lane_off = (lane / BS_LPU) * BS_UNIT_BYTES + (lane % BS_LPU) * (4 * BS_LW) + 8;  // the lane's window in a stage
  int cslot = 0;
  uint32_t parity = 0;
  for (int task = gw; task < p.tasks; task += nw) {
    const int u = task * BS_UPW + lane / BS_LPU;
    int img = 0, y0 = 0, x = 0, rows = p.R, nbytes = 0;  // nbytes <= 0: the lane is right of the image or its unit is past the last
    if (u < p.units) {
      img = u / per_img;
      const int rem = u - img * per_img;
      const int chunk = rem / p.ucols;
      x = (rem - chunk * p.ucols) * BS_UNIT + (lane % BS_LPU) * (4 * BS_LW);
      y0 = chunk * p.R;
      rows = min(p.R, p.nrows - y0);
      nbytes = min(4 * BS_LW, p.rowbytes - x);
    }
    const bool full = nbytes == 4 * BS_LW && p.vec_store;
    const bool clean = __all_sync(0xffffffffu, full);
    int min_rows = rows;  // the fewest output rows of the warp's units
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) min_rows = min(min_rows, __shfl_xor_sync(0xffffffffu, min_rows, o));

    uint32_t rE[BS_K][BS_LW], rO[BS_K][BS_LW], SE[BS_LW], SO[BS_LW];
#pragma unroll
    for (int q = 0; q < BS_LW; q++) {
      SE[q] = 0; SO[q] = 0;
#pragma unroll
      for (int j = 0; j < BS_K; j++) { rE[j][q] = 0; rO[j][q] = 0; }
    }

    // input row t of the task completes output row y0 + t - 4: drow is advanced once per input row, before its store
    unsigned char* drow = p.out_base[img] + (long long)(y0 - 5) * p.out_pitch + x;
    const long long pitch = p.out_pitch;
    for (int g = 0; g < p.groups; g++) {
      mbar_wait(&bars[cslot], parity);
      const unsigned char* st = ring + cslot * BS_STAGE_BYTES + lane_off;
      if (clean && g > 0 && BS_K * g < min_rows) {  // steady state: 5 rows of load, compute, store
#pragma unroll
        for (int j = 0; j < BS_K; j++) {
          box_stream_row<CS>(st + j * BS_BOXW, rE[j], rO[j], SE, SO, m256);
          drow += pitch;
          *reinterpret_cast<uint4*>(drow) = make_uint4(box_div_pack_hi(SE[0], SO[0], shl16), box_div_pack_hi(SE[1], SO[1], shl16),
                                                       box_div_pack_hi(SE[2], SO[2], shl16), box_div_pack_hi(SE[3], SO[3], shl16));
        }
      } else {
#pragma unroll
        for (int j = 0; j < BS_K; j++) {
          box_stream_row<CS>(st + j * BS_BOXW, rE[j], rO[j], SE, SO, m256);
          drow += pitch;
          const int t = BS_K * g + j;  // input row of the task (0 = image row y0 - 2)
          if (t >= 4 && t - 4 < rows && nbytes > 0) {
            uint32_t ow[BS_LW];
#pragma unroll
            for (int q = 0; q < BS_LW; q++) ow[q] = box_div_pack_hi(SE[q], SO[q], shl16);
            if (full)
              *reinterpret_cast<uint4*>(drow) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            else
              box_store_partial(drow, ow, nbytes);
          }
        }
      }
      __syncwarp();  // every lane is done reading the stage before TMA refills it
      if (lane < BS_UPW) produce();
      if (++cslot == BS_STAGES) { cslot = 0; parity ^= 1; }
    }
  }
}

static int layout_pitch(const vppb_img* i) {
  if (i->align <= 0) return -1;
  long long bs = (long long)i->border * i->elem_bytes;
  if (bs % i->align) bs += i->align - (bs % i->align);
  long long p = (long long)i->ncols * i->elem_bytes + 2 * bs;
  if (p % i->align) p += i->align - (p % i->align);
  return (int)p;
}

// TMA needs: library layout (so the bytes left/right of the domain belong to the row),
// 16-byte aligned pixel (0,0) and pitch, border >= 2 with at least 16 bytes of row before column 0.
static bool tma_eligible(const vppb_img* in) {
  if (in->align < 16 || in->border < 2) return false;
  if (((uintptr_t)in->base % 16) || (in->pitch % 16)) return false;
  if (layout_pitch(in) != in->pitch) return false;
  return true;
}

// rows per tile: 16 amortises the 4 halo rows better, 8 gives twice the CTAs (small frames cannot
// fill 148 SMs x 4 CTAs with 16-row tiles).  VPPB_BOX_TH=8|16 overrides for experiments.
static int box_tile_rows(int nrows, int rowbytes) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("VPPB_BOX_TH");
    forced = e ? atoi(e) : 0;
  }
  if (forced == 8 || forced == 16) return forced;
  const long long tiles16 = (long long)((rowbytes + BX_OUTW - 1) / BX_OUTW) * ((nrows + 15) / 16);
  return tiles16 >= 4LL * sm_count() ? 16 : 8;
}

// which byte kernel: VPPB_BOX_IMPL=tile selects the round-1 CTA tile kernels (kept for A/B timing), default = stream
static bool box_use_stream() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VPPB_BOX_IMPL");
    v = (e && !strcmp(e, "tile")) ? 0 : 1;
  }
  return v == 1;
}

// Rows per task: R = 5 m - 4 (a task then reads exactly m stages).  Small R = more tasks (parallelism for a single
// frame) but 4 extra input rows per task; pick the R with the smallest makespan estimate over the resident warps.
static int box_stream_rows(long long units_x_imgs, int nrows, int warps_per_sm, int* chunks_out) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("VPPB_BOX_R");
    forced = e ? atoi(e) : 0;
  }
  const long long warps = (long long)sm_count() * warps_per_sm;
  int best_r = 16;
  double best = 1e300;
  for (int m = 4; m <= 26; m++) {
    const int r = 5 * m - 4;
    if (forced > 0 && r != forced) continue;
    const long long chunks = (nrows + r - 1) / r, tasks = (chunks * units_x_imgs + BS_UPW - 1) / BS_UPW;
    const long long waves = (tasks + warps - 1) / warps;
    // per task: m stages of 5 rows + ~2 stages of pipeline fill when the warp starts; a wave costs its slowest warp
    const double cost = (double)waves * (5.0 * m + 2.0) + 10.0;
    if (cost < best) { best = cost; best_r = r; }
  }
  *chunks_out = (nrows + best_r - 1) / best_r;
  return best_r;
}

// n equally shaped, TMA-eligible images (n <= NB) in one launch of the streaming kernel
template <int CS, int NB>
static int box5_stream_launch_nb(const vppb_img* ins, const vppb_img* ups, const vppb_img* dns, const vppb_img* outs, int n, cudaStream_t st, const char* name) {
  const int rowbytes = ins[0].ncols * CS, nrows = ins[0].nrows;
  static std::atomic<unsigned long long> attr_done{0};
  int dev = 0;
  VPPB_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ULL << (dev & 63);
  if (!(attr_done.load(std::memory_order_acquire) & bit)) {
    VPPB_CUDA(cudaFuncSetAttribute(k_box5_stream<CS, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, BS_SMEM));
    attr_done.fetch_or(bit, std::memory_order_release);
  }
  BoxStream<NB> p;
  memset(&p, 0, sizeof(p));
  p.out_pitch = outs[0].pitch;
  p.nrows = nrows;
  p.rowbytes = rowbytes;
  p.ucols = (rowbytes + BS_UNIT - 1) / BS_UNIT;
  p.R = box_stream_rows((long long)p.ucols * n, nrows, BS_WARPS * BS_CTAS_PER_SM, &p.chunks);
  p.groups = (p.R + 4) / BS_K;
  p.vec_store = (((uintptr_t)outs[0].base % 16) == 0 && (outs[0].pitch % 16) == 0) ? 1 : 0;
  p.units = n * p.chunks * p.ucols;
  p.tasks = (p.units + BS_UPW - 1) / BS_UPW;
  p.one = 1u;
  const uint64_t width_el = ((uint64_t)rowbytes + 32 + 7) / 8;
  for (int k = 0; k < n; k++) {
    const vppb_img* in = &ins[k];
    unsigned char* origin = static_cast<unsigned char*>(in->base) - 2LL * in->pitch - 16;
    int rc = encode_tensor_map_2d(&p.maps[k], origin, CU_TENSOR_MAP_DATA_TYPE_UINT64, 8, width_el, (uint64_t)nrows + 4, (uint64_t)in->pitch,
                                  BS_BOXW / 8, BS_K);
    if (rc) return rc;
    p.out_base[k] = static_cast<unsigned char*>(outs[k].base);
    p.in_base[k] = static_cast<const unsigned char*>(in->base);
    p.up_base[k] = (ups && ups[k].base) ? static_cast<const unsigned char*>(ups[k].base) : nullptr;
    p.dn_base[k] = (dns && dns[k].base) ? static_cast<const unsigned char*>(dns[k].base) : nullptr;
  }
  {
    long long bs = (long long)ins[0].border * ins[0].elem_bytes;
    if (bs % ins[0].align) bs += ins[0].align - (bs % ins[0].align);
    p.in_pitch = ins[0].pitch;
    p.row_room = ins[0].pitch - (int)bs;
  }
  const int ctas = (p.tasks + BS_WARPS - 1) / BS_WARPS, resident = sm_count() * BS_CTAS_PER_SM;
  VPPB_CUDA(launch_dependent(k_box5_stream<CS, NB>, ctas < resident ? ctas : resident, BS_WARPS * 32, BS_SMEM, st, p));
  VPPB_LAUNCH_CHECK(name);
  return VPPB_OK;
}

// the kernel parameters carry one tensor map per image: a single image travels with a 1-entry block (launching a kernel
// with kilobytes of parameters costs microseconds), batches with up to 128
template <int CS>
static int box5_stream_launch(const vppb_img* ins, const vppb_img* ups, const vppb_img* dns, const vppb_img* outs, int n, cudaStream_t st, const char* name) {
  if (n == 1) return box5_stream_launch_nb<CS, 1>(ins, ups, dns, outs, n, st, name);
  if (n <= 4) return box5_stream_launch_nb<CS, 4>(ins, ups, dns, outs, n, st, name);
  if (n <= 32) return box5_stream_launch_nb<CS, 32>(ins, ups, dns, outs, n, st, name);
  return box5_stream_launch_nb<CS, BS_MAX_BATCH>(ins, ups, dns, outs, n, st, name);
}

template <int CS>
static int box5_bytes(const vppb_img* in, const vppb_img* out, void* stream, const char* name) {
  VPPB_REQUIRE(in && out && in->base && out->base, VPPB_E_ARG, "%s: NULL image", name);
  VPPB_REQUIRE(in->elem_bytes == CS && out->elem_bytes == CS, VPPB_E_ARG, "%s: element size must be %d", name, CS);
  VPPB_REQUIRE(same_domain(in, out), VPPB_E_ARG, "%s: domains differ", name);
  VPPB_REQUIRE(in->border >= 2, VPPB_E_BORDER, "%s: input border %d < 2", name, in->border);
  cudaStream_t st = as_stream(stream);
  const int rowbytes = in->ncols * CS;
  // one frame per launch: below ~8 tasks per resident warp the launch is dominated by fixed costs, where the CTA tile kernel
  // (one TMA box per CTA) is ~2 us cheaper; the per-warp streaming kernel wins as soon as the launch has real work (batches, 8K)
  static int single_policy = -1;
  if (single_policy < 0) {
    const char* e = getenv("VPPB_BOX_SINGLE");
    single_policy = (e && !strcmp(e, "stream")) ? 1 : 0;
  }
  const bool small = (long long)rowbytes * in->nrows < 96LL * 1024 * 1024;
  if (tma_eligible(in) && box_use_stream() && (single_policy == 1 || !small)) return box5_stream_launch<CS>(in, nullptr, nullptr, out, 1, st, name);
  if (tma_eligible(in)) {
    CUtensorMap tmap;
    unsigned char* origin = static_cast<unsigned char*>(in->base) - 2LL * in->pitch - 16;
    const uint64_t width_el = ((uint64_t)rowbytes + 32 + 7) / 8;
    const int th = box_tile_rows(in->nrows, rowbytes);
    int rc = encode_tensor_map_2d(&tmap, origin, CU_TENSOR_MAP_DATA_TYPE_UINT64, 8, width_el, (uint64_t)in->nrows + 4,
                                  (uint64_t)in->pitch, BX_BOXW / 8, th + 4);
    if (rc) return rc;
    const int strips = (rowbytes + BX_OUTW - 1) / BX_OUTW;
    const int row_tiles = (in->nrows + th - 1) / th;
    const int vec_store = (((uintptr_t)out->base % 16) == 0 && (out->pitch % 16) == 0) ? 1 : 0;
    // the opt-in shared-memory size is a per-device function attribute: set it once per device (bit = device ordinal)
    static std::atomic<unsigned long long> attr_done{0};
    int dev = 0;
    VPPB_CUDA(cudaGetDevice(&dev));
    const unsigned long long bit = 1ULL << (dev & 63);
    if (!(attr_done.load(std::memory_order_acquire) & bit)) {
      VPPB_CUDA(cudaFuncSetAttribute(k_box5_bytes_tma<CS, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, BoxCfg<16>::SMEM));
      VPPB_CUDA(cudaFuncSetAttribute(k_box5_bytes_tma<CS, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, BoxCfg<8>::SMEM));
      attr_done.fetch_or(bit, std::memory_order_release);
    }
    const int ntiles = strips * row_tiles;
    const int resident = sm_count() * (th == 16 ? 4 : 6);
    const int grid = ntiles < resident ? ntiles : resident;
    if (th == 16)
      VPPB_CUDA(launch_dependent(k_box5_bytes_tma<CS, 16>, grid, BX_THREADS, BoxCfg<16>::SMEM, st, tmap, view(out), rowbytes, strips, ntiles, vec_store, 1u));
    else
      VPPB_CUDA(launch_dependent(k_box5_bytes_tma<CS, 8>, grid, BX_THREADS, BoxCfg<8>::SMEM, st, tmap, view(out), rowbytes, strips, ntiles, vec_store, 1u));
  } else {
    long long total = (long long)in->nrows * rowbytes;
    long long blocks = (total + 255) / 256;
    long long cap = (long long)sm_count() * 16;
    k_box5_direct<unsigned char, int, CS><<<(int)(blocks < cap ? blocks : cap), 256, 0, st>>>(view(in), view(out), rowbytes);
  }
  VPPB_LAUNCH_CHECK(name);
  return VPPB_OK;
}

// A batch of equally shaped images in one launch per <= 32 images (k_box5_bytes_tma_batch).  Anything the batched
// kernel cannot take (mixed shapes, a view or an unaligned buffer among them) falls back to one launch per image -
// same results either way.
template <int CS>
static int box5_bytes_batch(const vppb_img* ins, const vppb_img* outs, int n, void* stream, const char* name) {
  VPPB_REQUIRE(ins && outs && n >= 0, VPPB_E_ARG, "%s: NULL batch", name);
  if (n == 0) return VPPB_OK;
  bool uniform = true;
  for (int i = 0; i < n; i++) {
    const vppb_img *in = &ins[i], *out = &outs[i];
    VPPB_REQUIRE(in->base && out->base, VPPB_E_ARG, "%s: NULL image %d", name, i);
    VPPB_REQUIRE(in->elem_bytes == CS && out->elem_bytes == CS, VPPB_E_ARG, "%s: element size must be %d (image %d)", name, CS, i);
    VPPB_REQUIRE(same_domain(in, out), VPPB_E_ARG, "%s: domains differ (image %d)", name, i);
    VPPB_REQUIRE(in->border >= 2, VPPB_E_BORDER, "%s: input border %d < 2 (image %d)", name, in->border, i);
    uniform = uniform && tma_eligible(in) && same_domain(in, &ins[0]) && out->pitch == outs[0].pitch &&
              (((uintptr_t)out->base % 16) == 0) == (((uintptr_t)outs[0].base % 16) == 0);
  }
  if (!uniform || n == 1) {
    for (int i = 0; i < n; i++) {
      int rc = box5_bytes<CS>(&ins[i], &outs[i], stream, name);
      if (rc) return rc;
    }
    return VPPB_OK;
  }
  cudaStream_t st = as_stream(stream);
  if (box_use_stream()) {
    for (int i0 = 0; i0 < n; i0 += BS_MAX_BATCH) {
      int rc = box5_stream_launch<CS>(ins + i0, nullptr, nullptr, outs + i0, std::min(BS_MAX_BATCH, n - i0), st, name);
      if (rc) return rc;
    }
    return VPPB_OK;
  }
  const int rowbytes = ins[0].ncols * CS, nrows = ins[0].nrows;
  const int strips = (rowbytes + BX_OUTW - 1) / BX_OUTW;
  // 16-row tiles (25 % halo rows instead of 50 %) as soon as the whole batch fills the machine with them
  const long long tiles16 = (long long)strips * ((nrows + 15) / 16) * std::min(n, BX_MAX_BATCH);
  const int th = tiles16 >= 4LL * sm_count() ? 16 : 8;
  const int row_tiles = (nrows + th - 1) / th, tpi = strips * row_tiles;
  const int vec_store = (((uintptr_t)outs[0].base % 16) == 0 && (outs[0].pitch % 16) == 0) ? 1 : 0;
  static std::atomic<unsigned long long> attr_done{0};
  int dev = 0;
  VPPB_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ULL << (dev & 63);
  if (!(attr_done.load(std::memory_order_acquire) & bit)) {
    VPPB_CUDA(cudaFuncSetAttribute(k_box5_bytes_tma_batch<CS, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, BoxCfg<16>::SMEM));
    VPPB_CUDA(cudaFuncSetAttribute(k_box5_bytes_tma_batch<CS, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, BoxCfg<8>::SMEM));
    attr_done.fetch_or(bit, std::memory_order_release);
  }
  const uint64_t width_el = ((uint64_t)rowbytes + 32 + 7) / 8;
  for (int i0 = 0; i0 < n; i0 += BX_MAX_BATCH) {
    const int m = std::min(BX_MAX_BATCH, n - i0);
    BoxBatch batch;
    memset(&batch, 0, sizeof(batch));
    for (int k = 0; k < m; k++) {
      const vppb_img* in = &ins[i0 + k];
      unsigned char* origin = static_cast<unsigned char*>(in->base) - 2LL * in->pitch - 16;
      int rc = encode_tensor_map_2d(&batch.maps[k], origin, CU_TENSOR_MAP_DATA_TYPE_UINT64, 8, width_el, (uint64_t)nrows + 4, (uint64_t)in->pitch,
                                    BX_BOXW / 8, th + 4);
      if (rc) return rc;
      batch.out_base[k] = static_cast<unsigned char*>(outs[i0 + k].base);
    }
    const long long total = (long long)m * tpi;
    const int resident = sm_count() * (th == 16 ? 4 : 6);
    const int grid = (int)(total < resident ? total : resident);
    if (th == 16)
      k_box5_bytes_tma_batch<CS, 16><<<grid, BX_THREADS, BoxCfg<16>::SMEM, st>>>(batch, m, outs[0].pitch, nrows, rowbytes, strips, tpi, vec_store, 1u);
    else
      k_box5_bytes_tma_batch<CS, 8><<<grid, BX_THREADS, BoxCfg<8>::SMEM, st>>>(batch, m, outs[0].pitch, nrows, rowbytes, strips, tpi, vec_store, 1u);
    VPPB_LAUNCH_CHECK(name);
  }
  return VPPB_OK;
}

// Row tiles: equally shaped TMA-eligible tiles; neighbours given per tile (base == NULL: none)
template <int CS>
static int box5_bytes_tiles(const vppb_img* ins, const vppb_img* ups, const vppb_img* dns, const vppb_img* outs, int n, void* stream, const char* name) {
  VPPB_REQUIRE(ins && outs && n >= 0, VPPB_E_ARG, "%s: NULL batch", name);
  for (int i = 0; i < n; i++) {
    const vppb_img *in = &ins[i], *out = &outs[i];
    VPPB_REQUIRE(in->base && out->base, VPPB_E_ARG, "%s: NULL image %d", name, i);
    VPPB_REQUIRE(in->elem_bytes == CS && out->elem_bytes == CS, VPPB_E_ARG, "%s: element size must be %d (image %d)", name, CS, i);
    VPPB_REQUIRE(same_domain(in, out) && same_domain(in, &ins[0]), VPPB_E_ARG, "%s: domains differ (image %d)", name, i);
    VPPB_REQUIRE(in->border >= 2 && in->nrows >= 2, VPPB_E_BORDER, "%s: tile %d needs border >= 2 and at least 2 rows", name, i);
    VPPB_REQUIRE(tma_eligible(in) && in->pitch == ins[0].pitch && in->border == ins[0].border && in->align == ins[0].align, VPPB_E_ARG,
                 "%s: tiles must share the library layout (image %d)", name, i);
    VPPB_REQUIRE(out->pitch == outs[0].pitch && (((uintptr_t)out->base % 16) == 0) == (((uintptr_t)outs[0].base % 16) == 0), VPPB_E_ARG,
                 "%s: outputs must share pitch and alignment (image %d)", name, i);
    for (const vppb_img* nb : {ups ? &ups[i] : nullptr, dns ? &dns[i] : nullptr})
      if (nb && nb->base)
        VPPB_REQUIRE(nb->pitch == in->pitch && nb->ncols == in->ncols && nb->nrows >= 2 && nb->elem_bytes == CS && nb->border == in->border &&
                         nb->align == in->align && ((uintptr_t)nb->base % 16) == 0,
                     VPPB_E_ARG, "%s: neighbour of tile %d must have the tile's layout", name, i);
    // the tile above contributes its LAST rows: they are addressed from its pixel (0,0) with ITS row count
    VPPB_REQUIRE(!(ups && ups[i].base) || ups[i].nrows == in->nrows, VPPB_E_ARG, "%s: the tile above tile %d must have as many rows (pass a sub-image of its last rows otherwise)", name, i);
  }
  cudaStream_t st = as_stream(stream);
  for (int i0 = 0; i0 < n; i0 += BS_MAX_BATCH) {
    int rc = box5_stream_launch<CS>(ins + i0, ups ? ups + i0 : nullptr, dns ? dns + i0 : nullptr, outs + i0, std::min(BS_MAX_BATCH, n - i0), st, name);
    if (rc) return rc;
  }
  return VPPB_OK;
}

}  // namespace vppb

using namespace vppb;

extern "C" {

int vppb_box5x5_u8c3_batch(const vppb_img* ins, const vppb_img* outs, int32_t n, void* stream) {
  return box5_bytes_batch<3>(ins, outs, n, stream, "vppb_box5x5_u8c3_batch");
}
int vppb_box5x5_u8_batch(const vppb_img* ins, const vppb_img* outs, int32_t n, void* stream) {
  return box5_bytes_batch<1>(ins, outs, n, stream, "vppb_box5x5_u8_batch");
}

int vppb_box5x5_u8c3_tiles(const vppb_img* ins, const vppb_img* ups, const vppb_img* downs, const vppb_img* outs, int32_t n, void* stream) {
  return box5_bytes_tiles<3>(ins, ups, downs, outs, n, stream, "vppb_box5x5_u8c3_tiles");
}
int vppb_box5x5_u8_tiles(const vppb_img* ins, const vppb_img* ups, const vppb_img* downs, const vppb_img* outs, int32_t n, void* stream) {
  return box5_bytes_tiles<1>(ins, ups, downs, outs, n, stream, "vppb_box5x5_u8_tiles");
}

int vppb_box5x5_u8c3(const vppb_img* in, const vppb_img* out, void* stream) {
  return box5_bytes<3>(in, out, stream, "vppb_box5x5_u8c3");
}

int vppb_box5x5_u8(const vppb_img* in, const vppb_img* out, void* stream) {
  return box5_bytes<1>(in, out, stream, "vppb_box5x5_u8");
}

int vppb_box5x5_i32(const vppb_img* in, const vppb_img* out, void* stream) {
  VPPB_REQUIRE(in && out && in->base && out->base, VPPB_E_ARG, "vppb_box5x5_i32: NULL image");
  VPPB_REQUIRE(in->elem_bytes == 4 && out->elem_bytes == 4, VPPB_E_ARG, "vppb_box5x5_i32: element size must be 4");
  VPPB_REQUIRE(same_domain(in, out), VPPB_E_ARG, "vppb_box5x5_i32: domains differ");
  VPPB_REQUIRE(in->border >= 2, VPPB_E_BORDER, "vppb_box5x5_i32: input border %d < 2", in->border);
  long long total = (long long)in->nrows * in->ncols;
  long long blocks = (total + 255) / 256;
  long long cap = (long long)sm_count() * 16;
  // int accumulation wraps like the reference's `int sum` on two's-complement hardware
  k_box5_direct<int, int, 1><<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(view(in), view(out), in->ncols);
  VPPB_LAUNCH_CHECK("vppb_box5x5_i32");
  return VPPB_OK;
}

}  // extern "C"
