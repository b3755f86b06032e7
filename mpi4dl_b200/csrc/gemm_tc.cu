// gemm_tc.cu -- tcgen05 (5th-gen tensor core) GEMM path for the 1x1 ("pointwise") convolutions
// that carry ~90% of the HBM traffic of the AmoebaNet-D / ResNet spatial stages (SURVEY 8d).
//
// NCHW makes a 1x1 convolution a plain GEMM per image with NO layout change:
//     fprop : Y[K x P] = W [K x C] * X [C x P]        P = H*W pixels, contiguous in memory
//     dgrad : dX[C x P] = W^T[C x K] * dY[K x P]
//     wgrad : dW[K x C] = dY[K x P] * X[C x P]^T       (reduction over pixels)
// fprop/dgrad: A = (padded) weights, K-major, TMA box {64 ch, 128 rows}, SWIZZLE_128B;
//              B = activations read IN PLACE by TMA as an MN-major operand: [ch][64 px] rows of 128 B,
//              SWIZZLE_128B; accumulator D[128 out-ch x BN px] lives in TMEM.  The epilogue goes
//              TMEM -> registers -> swizzled staging block in smem -> TMA store.
// wgrad:       both operands K-major straight from NCHW (pixels = reduction dim, contiguous).
// Box shapes:  a [64 ch][64 px] box touches 64 channel planes = 64 different 2 MB pages, and with plane strides
//              of 8..32 MB they alias in the translation cache: every 128 bytes cost a page walk (4.3 TB/s
//              ceiling, DESIGN.md "Address translation").  Layers with multi-page planes therefore move ONE
//              5-d box per stage, dims (64 px, 8 ch, P/64 px blocks, C/8 ch groups, image): the TMA unit walks
//              8 planes at a time and visits all pixel blocks of each before moving on; smem layout
//              [group][block][8 ch][128 B], which the UMMA descriptors express through LBO / SBO.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM alloc),
// warps 2..5 = epilogue.  Persistent CTAs, one per SM (wgrad for >= 400 input channels: CTA pairs, cta_group::2).
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace spc {

using namespace tc;

// conv_tap.cu: tap convolutions (stride 1, <= 128 output channels) without shifted copies
bool tap_v2_supported(int M, int Cin, int R, int S, int H, int W, int N, int stride);
int run_conv_tap_v2(const __nv_bfloat16* wp, int Mpad, int Cpad, const __nv_bfloat16* x, const __nv_bfloat16* bias,
                    __nv_bfloat16* y, int M, int Cin, int R, int S, int ph, int H, int W, int N, cudaStream_t st);

// wgrad_tap.cu: wgrad of the stride-1 tap convolutions (<= 128 channels on both sides), shifts formed in smem
bool wgrad_tap_supported(int K, int C, int R, int S, int H, int W, int stride);
int run_wgrad_tap(const __nv_bfloat16* x, const __nv_bfloat16* dy, float* dw, int K, int C, int N, int H, int W, int R, int S,
                  cudaStream_t st);

namespace {

constexpr int TC_THREADS = 192;
constexpr int A_BLK_BYTES = 128 * 128;      // one 128-row M block of A per stage (one 128-byte swizzle row per row): 16 KB
constexpr int TMEM_COLS = 512;

// Storage types of the tcgen05 GEMMs: bf16 (kind::f16) and fp32 read as TF32 (kind::tf32, opt-in, SPC_ALGO_TF32).
// One 128-byte swizzle row holds ROW = 64 bf16 or 32 fp32 elements: ROW channels per pipeline stage (K-major A), ROW
// pixels per B block (MN-major B) and per wgrad chunk.  One MMA reduces 32 bytes of K (16 bf16 / 8 TF32), so a stage is
// 4 MMA k-steps and every per-stage BYTE count is the same for both types; only the element counts per row change.
template <typename T> struct Tc;
template <> struct Tc<__nv_bfloat16> {
  static constexpr CUtensorMapDataType TMA_TYPE = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  // MN-major B operand (fprop / dgrad activations): TMA swizzle and matching UMMA descriptor layout
  static constexpr CUtensorMapSwizzle B_SWZ = CU_TENSOR_MAP_SWIZZLE_128B;
  static constexpr uint32_t B_LAYOUT = UMMA_SW128;
  static constexpr uint32_t B_SBO = 1024;   // 8-row swizzle atoms along K
  static __host__ __device__ constexpr uint32_t idesc(int M, int N, int a_mn, int b_mn) {
    return umma_idesc_bf16(M, N, a_mn, b_mn);
  }
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
    umma_bf16(d, a, b, id, acc);
  }
  static __device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16(v); }
  // 8 accumulator columns (+bias) -> one 16-byte chunk of the output row
  static __device__ __forceinline__ uint4 pack16(const uint32_t* r, float bias) {
    uint4 v;
    v.x = pack_bf16x2(__uint_as_float(r[0]) + bias, __uint_as_float(r[1]) + bias);
    v.y = pack_bf16x2(__uint_as_float(r[2]) + bias, __uint_as_float(r[3]) + bias);
    v.z = pack_bf16x2(__uint_as_float(r[4]) + bias, __uint_as_float(r[5]) + bias);
    v.w = pack_bf16x2(__uint_as_float(r[6]) + bias, __uint_as_float(r[7]) + bias);
    return v;
  }
};
template <> struct Tc<float> {
  static constexpr CUtensorMapDataType TMA_TYPE = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  // an MN-major TF32 operand is swizzled in 32-byte atoms (a 16-byte chunk holds only 4 fp32 values): four atoms per
  // 128-byte row, so the pattern repeats every 4 rows and one 8-channel MMA spans two 4-row K groups 512 B apart
  // (measured on B200, tools/tf32_mma_probe.cu, profiles/r3_tf32_mma_probe.txt).  K-major TF32 uses the plain swizzle.
  static constexpr CUtensorMapSwizzle B_SWZ = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
  static constexpr uint32_t B_LAYOUT = UMMA_SW128_ATOM32;
  static constexpr uint32_t B_SBO = 512;
  static __host__ __device__ constexpr uint32_t idesc(int M, int N, int a_mn, int b_mn) {
    return umma_idesc_tf32(M, N, a_mn, b_mn);
  }
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
    umma_tf32(d, a, b, id, acc);
  }
  static __device__ __forceinline__ float to_float(float v) { return v; }
  static __device__ __forceinline__ float from_float(float v) { return v; }
  // 4 accumulator columns (+bias) -> one 16-byte chunk of the output row, no rounding
  static __device__ __forceinline__ uint4 pack16(const uint32_t* r, float bias) {
    uint4 v;
    v.x = __float_as_uint(__uint_as_float(r[0]) + bias);
    v.y = __float_as_uint(__uint_as_float(r[1]) + bias);
    v.z = __float_as_uint(__uint_as_float(r[2]) + bias);
    v.w = __float_as_uint(__uint_as_float(r[3]) + bias);
    return v;
  }
};
template <typename T> constexpr int ROW = 128 / (int)sizeof(T);         // elements per 128-byte swizzle row
template <typename T> constexpr int KSTEP = 32 / (int)sizeof(T);        // K per MMA
template <typename T> constexpr int B_BLK_BYTES = ROW<T> * 128;         // [ROW ch][ROW px] block of B: 8 KB / 4 KB
constexpr int BK = ROW<__nv_bfloat16>;   // bf16-only paths (stride-2 dgrad repack, boundary GEMM workspace)

// ---- host: TMA descriptor encode (driver entry point fetched through the runtime) -------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// tensor map (bf16 unless told otherwise), rank <= 5; dims/strides innermost first (strides in BYTES for dims 1..).
int make_tmap_sw(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                 const uint32_t* box, CUtensorMapSwizzle swz, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return SPC_ECUDA;
  }
  // bind the primary context to this (possibly autograd worker) thread -- once per thread: cudaFree is not
  // allowed while a stream is being captured into a CUDA graph, and it is not free either
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    if (cudaFree(nullptr) != cudaSuccess) {
      set_error("tcgen05 conv: no CUDA context on this thread");
      return SPC_ECUDA;
    }
    ctx_bound = true;
  }
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gs[i - 1] = strides_bytes[i];
  }
  CUresult r = enc(m, dt, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rank=%d dims=[%llu,%llu,%llu] strides=[%llu,%llu]", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 1 ? strides_bytes[1] : 0),
              (unsigned long long)(rank > 2 ? strides_bytes[2] : 0));
    return SPC_ECUDA;
  }
  return SPC_OK;
}

int make_tmap(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  return make_tmap_sw(m, base, rank, dims, strides_bytes, box, CU_TENSOR_MAP_SWIZZLE_128B, dt);
}

// ---- weight repack: Wp[tap][m][c] (zero padded to [taps][Mpad][Cpad]) ------------------------------
// element = w[m*sm + c*sc + (flip ? taps-1-tap : tap)]
//   fprop: m = out channel k, c = in channel:  sm = C*RS, sc = RS, flip = 0     (w is [K][C][R][S])
//   dgrad: m = c, c = k (transposed) and the filter is rotated by 180 degrees:  sm = RS, sc = C*RS, flip = 1
template <typename T>
__global__ void repack_weights_kernel(const T* __restrict__ w, T* __restrict__ wp, int M,
                                      int Cc, int Mpad, int Cpad, int taps, long long sm, long long sc, int flip) {
  const int total = taps * Mpad * Cpad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c = i % Cpad;
    const int m = (i / Cpad) % Mpad;
    const int tap = i / (Cpad * Mpad);
    T v = Tc<T>::from_float(0.f);
    if (m < M && c < Cc) v = w[(size_t)m * sm + (size_t)c * sc + (flip ? taps - 1 - tap : tap)];
    wp[i] = v;
  }
}

// ---- fprop / dgrad kernel -----------------------------------------------------------------------
constexpr int BN_DEFAULT = 128;               // pixels per tile (two 64-pixel swizzle blocks); 256 in the wide-N variant
// epilogue staging: one 128-channel block of 128 pixels of a tile (32 KB bf16, 64 KB fp32)
template <typename T> constexpr int OUT_BUF_BYTES = 128 * 128 * (int)sizeof(T);
constexpr int MAX_STAGES = 8;

struct PwParams {
  int M;                       // valid output channels
  int Cin;                     // reduction length (input channels)
  int P;                       // pixels per image
  int N;                       // images
  int tiles_per_image;
  int num_mg;                  // groups of MB*128 output channels (X tile re-read per group, from L2)
  int num_tiles;               // N * tiles_per_image * num_mg
  int stages;                  // pipeline depth (runtime, <= MAX_STAGES)
  int wres;                    // 1: all weight chunks stay resident in smem (loaded once per CTA)
  int out_bufs;                // 1 or 2 epilogue staging buffers
  int taps, S, ph, pw;         // filter taps (R*S), filter width, zero padding (tap mode)
  int W, Mpad;                 // image width (tap mode: tiles are 64-pixel row segments), padded M
  int shiftN;                  // N when the activations are S column-shifted copies, else 0
  int rowmul;                  // input row = rowmul * output row + tap row offset (2 for stride-2 convs)
  int tgroup;                  // consecutive tiles handled back-to-back by one CTA (DRAM page locality)
  const void* bias;            // [M] or null, storage type
  void* y;                     // output base [N][M][P] (coalesced-store epilogue)
  int epi_stg;                 // 1: staged tile leaves with per-thread 16-B stores (full 128-B lines), 0: TMA store
  int x5, y5;                  // 1: activations / outputs move as ONE 5-d box per tile whose traversal order is
                               // (8-channel group, 64-pixel block, channel, pixel): the TMA unit touches 8 channel
                               // planes (2 MB pages each) at a time and visits both pixel blocks of each before moving
                               // on, instead of walking 64 / 128 planes per pixel block (address-translation reach)
  int stationary_ok;           // host: stationary weights allowed with several output-channel groups
  int xbox, ybox;              // channel rows per TMA load / store box (64 / 128 = one box per 64-pixel block; smaller
                               // boxes walk FEWER channel planes -- 2 MB pages -- between the two pixel blocks of a tile)
};

// EXT = false compiles the round-2 options (5-d boxes, box-row knobs, per-thread-store epilogue) out: the launches that
// use none of them (every tap-mode launch; the stem is epilogue-bound and ran 16 % slower with the extra branches in
// its epilogue, A/B on one GPU) get exactly the plain kernel.  T = float (TF32 operands) is only built with EXT = false.
template <typename T, int MB, int BN, bool EXT>
__global__ void __launch_bounds__(TC_THREADS, 1)
pw_gemm_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
               const __grid_constant__ CUtensorMap tmap_x4, const __grid_constant__ CUtensorMap tmap_y,
               const PwParams p) {
  constexpr int BK = ROW<T>;               // channels per pipeline stage (one 128-byte swizzle row of A)
  constexpr int PXB = ROW<T>;              // pixels per B block (one 128-byte swizzle row of B)
  constexpr int KS = KSTEP<T>;
  constexpr int BBLK = B_BLK_BYTES<T>;
  constexpr int OUTB = OUT_BUF_BYTES<T>;
  constexpr int NB = BN / PXB;
  constexpr int ACC = (MB <= 2) ? 2 : 1;
  static_assert(ACC * MB * BN <= TMEM_COLS, "TMEM budget");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int kchunks = (p.Cin + BK - 1) / BK;
  const int ksteps_total = (p.Cin + KS - 1) / KS;
  const int iters = p.taps * kchunks;      // K loop: (filter tap, BK-channel chunk)
  const int wres_bytes = p.wres ? iters * MB * A_BLK_BYTES : 0;
  const int stage_bytes = (p.wres ? 0 : MB * A_BLK_BYTES) + NB * BBLK;
  uint8_t* wres = smem;
  uint8_t* stage0 = smem + wres_bytes;
  uint8_t* outbuf = stage0 + p.stages * stage_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(outbuf + p.out_bufs * OUTB);
  uint64_t* empty = full + MAX_STAGES;
  uint64_t* tfull = empty + MAX_STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* wfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool x5 = EXT && p.x5, y5 = EXT && p.y5, epi_stg = EXT && p.epi_stg;
  const int xbox = EXT ? p.xbox : BK, ybox = EXT ? p.ybox : 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < ACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 128); }
    mbar_init(wfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      tma_prefetch_desc(&tmap_w);
      tma_prefetch_desc(&tmap_x);
      if (p.wres) {
        // weights-stationary: the CTA keeps the (padded) filter rows of ITS group of output channels in smem for its
        // whole life.  With several groups the grid is a multiple of num_mg, so tile t = it * grid + blockIdx.x
        // always lands in group blockIdx.x % num_mg (t % num_mg below), and the CTAs of the other groups read the same
        // activation tile at about the same time (L2 hits).
        const int mg0 = blockIdx.x % p.num_mg;
        mbar_arrive_expect_tx(wfull, wres_bytes);
        for (int it = 0; it < iters; ++it)
#pragma unroll
          for (int mb = 0; mb < MB; ++mb)
            tma_load_2d(wres + (it * MB + mb) * A_BLK_BYTES, &tmap_w, wfull, (it % kchunks) * BK,
                        (it / kchunks) * p.Mpad + mg0 * (MB * 128) + mb * 128);
      }
      int s = 0, ph = 0;
      for (int it = 0;; ++it) {
        const int t = ((it / p.tgroup) * gridDim.x + blockIdx.x) * p.tgroup + it % p.tgroup;
        if ((it / p.tgroup) * gridDim.x * p.tgroup >= p.num_tiles) break;
        if (t >= p.num_tiles) continue;
        const int mg = t % p.num_mg;
        const int tt = t / p.num_mg;
        const int n = tt / p.tiles_per_image;
        const int p0 = (tt % p.tiles_per_image) * BN;
        for (int it = 0; it < iters; ++it) {
          const int kc = it % kchunks, tap = it / kchunks;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = stage0 + s * stage_bytes;
          mbar_arrive_expect_tx(&full[s], stage_bytes);
          if (!p.wres) {
#pragma unroll
            for (int mb = 0; mb < MB; ++mb)
              tma_load_2d(st + mb * A_BLK_BYTES, &tmap_w, &full[s], kc * BK, tap * p.Mpad + mg * (MB * 128) + mb * 128);
            st += MB * A_BLK_BYTES;
          }
          if (p.taps == 1) {
            if (x5) {
              tma_load_5d(st, &tmap_x, &full[s], 0, 0, p0 >> 6, kc * (BK / 8), n);
            } else if (xbox == BK) {
#pragma unroll
              for (int j = 0; j < NB; ++j) tma_load_3d(st + j * BBLK, &tmap_x, &full[s], p0 + j * PXB, kc * BK, n);
            } else {
              for (int cg = 0; cg < BK; cg += xbox)
#pragma unroll
                for (int j = 0; j < NB; ++j)
                  tma_load_3d(st + j * BBLK + cg * 128, &tmap_x, &full[s], p0 + j * PXB, kc * BK + cg, n);
            }
          } else {
            // shifted window of this tap; out-of-image rows / columns are zero-filled by TMA (= zero padding)
            const int dr = tap / p.S - p.ph;
            const int img = n + (tap % p.S) * p.shiftN;   // column shift = which pre-shifted copy
#pragma unroll
            for (int j = 0; j < NB; ++j) {
              const int q = p0 + j * PXB, hq = q / p.W, wq = q - hq * p.W;
              tma_load_4d(st + j * BBLK, &tmap_x4, &full[s], wq, hq * p.rowmul + dr, kc * BK, img);
            }
          }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      constexpr uint32_t IDESC = Tc<T>::idesc(128, BN, /*a_mn=*/0, /*b_mn=*/1);
      if (p.wres) { mbar_wait(wfull, 0); tc_fence_after(); }
      int s = 0, ph = 0, a = 0, aph = 0;
      for (int it = 0;; ++it) {
        const int t = ((it / p.tgroup) * gridDim.x + blockIdx.x) * p.tgroup + it % p.tgroup;
        if ((it / p.tgroup) * gridDim.x * p.tgroup >= p.num_tiles) break;
        if (t >= p.num_tiles) continue;
        mbar_wait(&tempty[a], aph ^ 1);
        tc_fence_after();
        for (int it = 0; it < iters; ++it) {
          const int kc = it % kchunks;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t st = smem_u32(stage0 + s * stage_bytes);
          const uint32_t sa = p.wres ? smem_u32(wres + it * MB * A_BLK_BYTES) : st;
          const uint32_t sb = p.wres ? st : st + MB * A_BLK_BYTES;
          const int nsteps = min(4, ksteps_total - kc * 4);
          for (int ks = 0; ks < nsteps; ++ks) {
            // B: MN-major SW128. KS channels = KS rows of 128 B (K groups at SBO); PXB-px blocks at LBO = BBLK
            // (bf16: 16 channels = two 8-row groups, 64-px blocks at 8 KB; TF32: 8 channels = two 4-row groups of
            // 32-byte atoms, 32-px blocks at 4 KB)
            // (5-d box layout [8-ch group][px block][8 ch][128 B]: px blocks at LBO = 1 KB, channel groups at SBO = 2 KB)
            const uint64_t bdesc = x5 ? umma_desc(sb + ks * (NB * 2048), 1024, NB * 1024)
                                        : umma_desc(sb + ks * (KS * 128), BBLK, Tc<T>::B_SBO, Tc<T>::B_LAYOUT);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
              // A: K-major SW128. 8-row groups at SBO = 1024 B; +32 B per k-step
              const uint64_t adesc = umma_desc(sa + mb * A_BLK_BYTES + ks * 32, 16, 1024);
              Tc<T>::mma(tmem_base + (a * MB + mb) * BN, adesc, bdesc, IDESC, (it | ks) ? 1u : 0u);
            }
          }
          umma_commit(&empty[s]);
          if (it == iters - 1) umma_commit(&tfull[a]);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        if (++a == ACC) { a = 0; aph ^= 1; }
      }
    }
  } else {
    // ===== epilogue: TMEM -> registers -> swizzled smem -> TMA store of [128 ch][64 px] boxes =====
    const int quarter = warp & 3;          // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;   // row of the 128-channel block (= TMEM lane)
    const bool leader = (threadIdx.x == 64);
    int a = 0, aph = 0, ob = 0;
    for (int it = 0;; ++it) {
      const int t = ((it / p.tgroup) * gridDim.x + blockIdx.x) * p.tgroup + it % p.tgroup;
      if ((it / p.tgroup) * gridDim.x * p.tgroup >= p.num_tiles) break;
      if (t >= p.num_tiles) continue;
      const int mg = t % p.num_mg;
      const int tt = t / p.num_mg;
      const int n = tt / p.tiles_per_image;
      const int p0 = (tt % p.tiles_per_image) * BN;
      mbar_wait(&tfull[a], aph);
      tc_fence_after();
#pragma unroll 1
      for (int mb = 0; mb < MB; ++mb) {
        const int k0 = mg * (MB * 128) + mb * 128;
        if (k0 >= p.M) break;                       // block-uniform: nothing valid in this block
        const int k = k0 + row;
        const float bias = (k < p.M && p.bias) ? Tc<T>::to_float(static_cast<const T*>(p.bias)[k]) : 0.f;
#pragma unroll 1
        for (int h = 0; h < BN / 128; ++h) {        // 128 pixels (128 / PXB blocks) of the tile at a time
          const int ph0 = p0 + h * 128;
          uint8_t* buf = outbuf + ob * OUTB;
          if (epi_stg) {
            // every thread has copied the previous contents of this buffer out (with two buffers the barrier of the
            // block in between already guarantees that)
            if (p.out_bufs == 1) named_bar_sync(1, 128);
          } else {
            // the TMA store that last read this buffer must have finished reading it
            if (leader) { if (p.out_bufs == 2) tma_store_wait_read<1>(); else tma_store_wait_read<0>(); }
            named_bar_sync(1, 128);
          }
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (a * MB + mb) * BN + h * 128 + cc * 32, r);
            tmem_ld_wait();
            constexpr int EPC = 16 / (int)sizeof(T);   // elements per 16-byte chunk
#pragma unroll
            for (int q = 0; q < 32 / EPC; ++q) {
              const int e = cc * (32 / EPC) + q;       // 16-B chunk of this channel row: block e / 8, chunk e % 8
              uint8_t* blk = y5 ? buf + (row >> 3) * 2048 + (e >> 3) * 1024 + (row & 7) * 128
                                  : buf + (e >> 3) * (128 * 128) + row * 128;
              const uint4 v = Tc<T>::pack16(r + EPC * q, bias);
              const int chunk = (e & 7) ^ (row & 7);   // SWIZZLE_128B: 16-B chunk ^ (row % 8)
              *reinterpret_cast<uint4*>(blk + chunk * 16) = v;
            }
          }
          if (h == BN / 128 - 1 && (mb == MB - 1 || k0 + 128 >= p.M)) {   // last read of this tile's accumulators
            tc_fence_before();
            mbar_arrive(&tempty[a]);
          }
          if (epi_stg) {
            // staged [128 ch][2 x 64 px] tile -> global: 8 consecutive threads write one full 128-B line of a channel
            // row, so every store instruction of a warp fills 4 whole lines.  Nothing waits for the writes to land:
            // the staging buffer is free again as soon as it has been read, and the TMA unit only serves the loads.
            named_bar_sync(1, 128);
            const int et = threadIdx.x - 64, g = et & 7, r0 = et >> 3;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int px = ph0 + j * 64 + g * 8;
              if (px < p.P) {
#pragma unroll
                for (int rr = 0; rr < 8; ++rr) {
                  const int rw = rr * 16 + r0;
                  if (k0 + rw < p.M) {
                    const uint4 v = *reinterpret_cast<const uint4*>(buf + j * (128 * 128) + rw * 128 + ((g ^ (rw & 7)) << 4));
                    __stcs(reinterpret_cast<uint4*>(static_cast<T*>(p.y) + ((size_t)n * p.M + k0 + rw) * p.P + px), v);
                  }
                }
              }
            }
          } else {
            fence_proxy_async();        // make the smem writes visible to the TMA (async proxy)
            named_bar_sync(1, 128);
            if (leader) {
              if (y5) {
                tma_store_5d(&tmap_y, buf, 0, 0, ph0 >> 6, k0 >> 3, n);
              } else if (ybox == 128) {
#pragma unroll
                for (int j = 0; j < 128 / PXB; ++j) tma_store_3d(&tmap_y, buf + j * (128 * 128), ph0 + j * PXB, k0, n);
              } else {
                for (int cg = 0; cg < 128 && k0 + cg < p.M; cg += ybox)
#pragma unroll
                  for (int j = 0; j < 128 / PXB; ++j)
                    tma_store_3d(&tmap_y, buf + j * (128 * 128) + cg * 128, ph0 + j * PXB, k0 + cg, n);
              }
              tma_store_commit();
            }
          }
          if (p.out_bufs == 2) ob ^= 1;
        }
      }
      if (++a == ACC) { a = 0; aph ^= 1; }
    }
    if (leader && !epi_stg) tma_store_wait_read<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
// tuning knob: positive integer from the environment, else `dflt` (tools/wgrad_probe.py sweeps these)
// Every knob is read from the environment ONCE per process (getenv on the launch path showed up in the
// N=8 step, which is CPU-bound): a small table keyed by the name's address (names are string literals).
struct EnvKnob { const char* name; const char* val; };
EnvKnob g_env_tab[32];
int g_env_n = 0;
inline const char* env_get(const char* name) {
  for (int i = 0; i < g_env_n; ++i)
    if (g_env_tab[i].name == name) return g_env_tab[i].val;
  const char* v = getenv(name);
  if (g_env_n < 32) { g_env_tab[g_env_n].name = name; g_env_tab[g_env_n].val = v; ++g_env_n; }
  return v;
}
inline int env_int(const char* name, int dflt) {
  const char* e = env_get(name);
  const int v = e ? atoi(e) : 0;
  return v > 0 ? v : dflt;
}
inline int sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

constexpr int SMEM_LIMIT = 222 * 1024;   // leave room for a small co-resident kernel (halo post/collect, boundary strips)
constexpr int SMEM_AUX = 1024 /*align*/ + 512 /*barriers*/;

template <typename T, int MB, int BN, bool EXT>
int launch_pw_ext(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& tx4, const CUtensorMap& ty, PwParams p,
              cudaStream_t st) {
  constexpr int OUTB = OUT_BUF_BYTES<T>;
  const int kchunks = (p.Cin + ROW<T> - 1) / ROW<T>;
  const int budget = SMEM_LIMIT - SMEM_AUX;
  const int wres_bytes = p.taps * kchunks * MB * A_BLK_BYTES;
  const int sms = sm_count();
  int grid = p.num_tiles < sms ? p.num_tiles : sms;
  if (p.num_tiles < 16 * sms) p.tgroup = 1;   // small problems: keep every SM busy
  // resident filter rows: up to 128 KB with bf16; fp32 (64 KB staging buffer) keeps room for 3 activation stages
  const int wres_max = sizeof(T) == 2 ? 128 * 1024 : budget - OUTB - 3 * (BN / ROW<T>) * B_BLK_BYTES<T>;
  // stationary weights with several groups of output channels: every CTA serves one group (see the kernel), which needs
  // a grid that is a multiple of num_mg and tiles dealt round-robin
  bool stationary = wres_bytes <= wres_max;
  if (stationary && p.num_mg > 1) {
    if (p.stationary_ok && grid >= 4 * p.num_mg) { grid = grid / p.num_mg * p.num_mg; p.tgroup = 1; }
    else stationary = false;
  }
  p.wres = stationary ? 1 : 0;
  const int stage_bytes = (p.wres ? 0 : MB * A_BLK_BYTES) + (BN / ROW<T>) * B_BLK_BYTES<T>;
  const int rem = budget - (p.wres ? wres_bytes : 0);
  p.out_bufs = 2;
  p.stages = (rem - 2 * OUTB) / stage_bytes;
  if (p.stages < 3 || env_int("SPC_PW_OUTBUFS", 2) == 1) { p.out_bufs = 1; p.stages = (rem - OUTB) / stage_bytes; }
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  SPC_REQUIRE(p.stages >= 2, "tcgen05 conv: shared memory budget too small (MB=%d kchunks=%d)", MB, kchunks);
  const int smem = (p.wres ? wres_bytes : 0) + p.stages * stage_bytes + p.out_bufs * OUTB + SMEM_AUX;
  auto kern = pw_gemm_kernel<T, MB, BN, EXT>;
  static bool attr_set = false;   // per instantiation
  if (!attr_set) {
    SPC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set = true;
  }
  kern<<<grid, TC_THREADS, smem, st>>>(tw, tx, tx4, ty, p);
  count_launch();
  SPC_CHECK_CUDA(cudaGetLastError());
  return SPC_OK;
}

template <typename T, int MB, int BN>
int launch_pw(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& tx4, const CUtensorMap& ty, const PwParams& p,
              cudaStream_t st) {
  if constexpr (sizeof(T) == 4) {   // TF32 launches use none of the round-2 options (run_conv_tc)
    return launch_pw_ext<T, MB, BN, false>(tw, tx, tx4, ty, p, st);
  } else {
    const bool ext = p.x5 || p.y5 || p.epi_stg || p.xbox != ROW<T> || p.ybox != 128;
    return ext ? launch_pw_ext<T, MB, BN, true>(tw, tx, tx4, ty, p, st)
               : launch_pw_ext<T, MB, BN, false>(tw, tx, tx4, ty, p, st);
  }
}

// [N][Cc][P] activations, boxes of one 128-byte row of pixels (64 bf16 / 32 fp32) x box_rows channels
template <typename T>
int make_act_tmap(CUtensorMap* m, const void* base, int P, int Cc, int N, int box_rows,
                  CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  const uint64_t dims[3] = {(uint64_t)P, (uint64_t)Cc, (uint64_t)N};
  const uint64_t strides[3] = {0, (uint64_t)P * sizeof(T), (uint64_t)P * Cc * sizeof(T)};
  const uint32_t box[3] = {(uint32_t)ROW<T>, (uint32_t)box_rows, 1};
  return make_tmap_sw(m, base, 3, dims, strides, box, swz, Tc<T>::TMA_TYPE);
}

// [N][Cc][P] bf16 as (64 px, 8 channels, P/64 pixel blocks, Cc/8 channel groups, N): one box = `groups` channel
// groups x `blocks` pixel blocks, laid out in shared memory as [group][block][8 ch][128 B]
int make_act_tmap5(CUtensorMap* m, const void* base, int P, int Cc, int N, int groups, int blocks) {
  const uint64_t dims[5] = {64, 8, (uint64_t)P / 64, (uint64_t)Cc / 8, (uint64_t)N};
  const uint64_t strides[5] = {0, (uint64_t)P * 2, 128, (uint64_t)P * 16, (uint64_t)P * Cc * 2};
  const uint32_t box[5] = {64, 8, (uint32_t)blocks, (uint32_t)groups, 1};
  return make_tmap(m, base, 5, dims, strides, box);
}

template <typename T>
int launch_shift_copies(const void* x, void* xs, size_t planes, int H, int W, int S, int pw, int cs, cudaStream_t st);

// Geometry of one tcgen05 convolution launch (fprop, or dgrad expressed as a convolution of dY).
template <typename T>
struct TcConv {
  const T* w;                  // original filter [K][C][R][S]
  long long sm, sc;            // strides of (output channel m, reduction channel c) in w
  int flip;                    // rotate taps by 180 degrees (dgrad)
  int M, Cin;                  // output channels, reduction channels
  int R, S, ph, pw;            // filter and zero padding
  int H, W, N;                 // input image
  int stride;                  // 1 or 2 (both axes)
  const T* prepacked;          // if set: weights already in [taps][Mpad][Cpad] layout (1024-aligned)
};

// Y[N][M][H*W] = sum_taps Wp[tap][M x Cin] * shift_tap(X[N][Cin][H][W])  (+bias)
// T = float: TF32 operands; tap convolutions always go through the shifted copies (conv_tap.cu is bf16-only) and none
// of the bf16 tuning knobs apply.
template <typename T>
int run_conv_tc(const TcConv<T>& c, const T* x, const T* bias, T* y, void* ws, size_t ws_bytes, cudaStream_t st) {
  constexpr bool BF = sizeof(T) == 2;
  constexpr int BK = ROW<T>;
  constexpr size_t ES = sizeof(T);
  const int taps = c.R * c.S;
  const int cs = c.stride;
  const int Ho = c.H / cs, Wo = c.W / cs;
  const int Pin = c.H * c.W, P = Ho * Wo;            // P: output pixels per image
  const int Mpad = round_up(c.M, 128), Cpad = round_up(c.Cin, BK);
  const bool v2 = BF && taps > 1 && !env_get("SPC_TAP_V1") && tap_v2_supported(c.M, c.Cin, c.R, c.S, c.H, c.W, c.N, cs);
  const bool copies = (c.S > 1 || cs > 1) && taps > 1 && !v2;   // column-shifted (and subsampled) copies of the input
  const uintptr_t ws0 = reinterpret_cast<uintptr_t>(ws);
  const uintptr_t wp_addr = (ws0 + 1023) & ~(uintptr_t)1023;
  const size_t wp_bytes = c.prepacked ? 0 : (size_t)taps * Mpad * Cpad * ES;
  const uintptr_t xs_addr = (wp_addr + wp_bytes + 1023) & ~(uintptr_t)1023;
  const size_t xs_bytes = copies ? (size_t)c.S * c.N * c.Cin * c.H * Wo * ES : 0;
  const size_t need = (xs_addr - ws0) + xs_bytes;
  SPC_REQUIRE((ws && ws_bytes >= need) || need <= 1024, "tcgen05 conv: workspace too small (%zu < %zu)", ws_bytes, need);
  const T* wp = c.prepacked;
  if (!c.prepacked) {
    T* wpm = reinterpret_cast<T*>(wp_addr);
    const int total = taps * Mpad * Cpad;
    int blocks = (total + 255) / 256;
    if (blocks > 1184) blocks = 1184;
    repack_weights_kernel<T><<<blocks, 256, 0, st>>>(c.w, wpm, c.M, c.Cin, Mpad, Cpad, taps, c.sm, c.sc, c.flip);
    count_launch();
    SPC_CHECK_CUDA(cudaGetLastError());
    wp = wpm;
  }
  if constexpr (BF) {
    if (v2) return run_conv_tap_v2(wp, Mpad, Cpad, x, bias, y, c.M, c.Cin, c.R, c.S, c.ph, c.H, c.W, c.N, st);
  }
  const T* xsrc = x;
  if (copies) {
    void* xs = reinterpret_cast<void*>(xs_addr);
    int rc0 = launch_shift_copies<T>(x, xs, (size_t)c.N * c.Cin, c.H, c.W, c.S, c.pw, cs, st);
    if (rc0) return rc0;
    xsrc = reinterpret_cast<const T*>(xs);
  }
  CUtensorMap tw, tx, tx4, ty;
  // Wide-N variant (256-pixel tiles, one 128-row block of output channels per CTA with its filter rows resident in
  // shared memory, double-buffered accumulators): for pointwise layers with 3+ blocks of output channels and 256..512
  // input channels, which are bound by the tensor pipe -- a 128x128x16 MMA costs almost what a 128x256x16 one does
  // (measured 185-270 vs 222 clk), so N = 256 should nearly halve the MMA time per pixel.  MEASURED (profiles/
  // r2h_pw_n256.txt): slower, 416->416 @1024^2 0.56 -> 0.65 ms -- with the filter rows resident only two 32 KB
  // activation stages fit, and 64 KB in flight per SM at ~2 us of load latency caps the CTA at ~35 GB/s.  Kept behind
  // SPC_PW_N256=1 (off by default); results are bit-identical to the default path.
  const char* n256_env = env_get("SPC_PW_N256");
  const bool n256 = BF && taps == 1 && cs == 1 && Mpad / 128 >= 3 && (Cpad / BK) * A_BLK_BYTES <= 128 * 1024 &&
                    P % 256 == 0 && (n256_env ? atoi(n256_env) != 0 : false);
  const int BN = n256 ? 256 : BN_DEFAULT;
  int xbox = (BF && taps == 1) ? env_int("SPC_PW_XBOX", BK) : BK, ybox = BF ? env_int("SPC_PW_YBOX", 128) : 128;
  if (xbox != 8 && xbox != 16 && xbox != 32) xbox = BK;
  if (ybox != 8 && ybox != 16 && ybox != 32 && ybox != 64) ybox = 128;
  // 5-d boxes (see PwParams::x5): measured on B200 (profiles/r2f_pw_box5.txt) +20..32 % on the layers whose channel
  // planes span several 2 MB pages (104->208 @4096^2: 4.30 -> 5.67 TB/s), neutral at 1024^2 planes -> on from 4 MB planes.
  // SPC_PW_BOX5 = 0..3 overrides (bit 0: activations, bit 1: outputs).  bf16 only.
  const char* box5_env = env_get("SPC_PW_BOX5");
  const int box5 = !BF ? 0 : box5_env ? atoi(box5_env) : ((size_t)P * 2 >= ((size_t)4 << 20) ? 3 : 0);
  const int x5 = (taps == 1 && cs == 1 && (box5 & 1) && P % 64 == 0 && c.Cin % 8 == 0 && xbox == BK) ? 1 : 0;
  const int y5 = (taps == 1 && (box5 & 2) && P % 64 == 0 && c.M % 8 == 0 && ybox == 128) ? 1 : 0;
  {
    const uint64_t dims[2] = {(uint64_t)Cpad, (uint64_t)taps * Mpad};
    const uint64_t strides[2] = {0, (uint64_t)Cpad * ES};
    const uint32_t box[2] = {(uint32_t)BK, 128};
    int rc = make_tmap(&tw, wp, 2, dims, strides, box, Tc<T>::TMA_TYPE);
    if (rc) return rc;
  }
  int rc;
  if (taps > 1) {
    // (copies of) the input as [img][Cin][H][Wo]; img = n + s*N for the copy of filter column s
    const uint64_t dims[4] = {(uint64_t)Wo, (uint64_t)c.H, (uint64_t)c.Cin, (uint64_t)c.N * (copies ? c.S : 1)};
    const uint64_t strides[4] = {0, (uint64_t)Wo * ES, (uint64_t)c.H * Wo * ES, (uint64_t)c.H * Wo * c.Cin * ES};
    const uint32_t box[4] = {(uint32_t)ROW<T>, 1, (uint32_t)BK, 1};
    rc = make_tmap_sw(&tx4, xsrc, 4, dims, strides, box, Tc<T>::B_SWZ, Tc<T>::TMA_TYPE);
    if (rc) return rc;
    tx = tx4;
  } else {
    rc = x5 ? make_act_tmap5(&tx, x, Pin, c.Cin, c.N, BK / 8, BN / 64)
            : make_act_tmap<T>(&tx, x, Pin, c.Cin, c.N, xbox, Tc<T>::B_SWZ);
    if (rc) return rc;
    tx4 = tx;
  }
  rc = y5 ? make_act_tmap5(&ty, y, P, c.M, c.N, 16, 2) : make_act_tmap<T>(&ty, y, P, c.M, c.N, ybox);
  if (rc) return rc;
  PwParams p{};
  p.xbox = xbox; p.ybox = ybox; p.x5 = x5; p.y5 = y5;
  p.bias = bias; p.M = c.M; p.Cin = c.Cin; p.P = P; p.N = c.N;
  p.taps = taps; p.S = c.S; p.ph = c.ph; p.pw = c.pw; p.W = Wo; p.Mpad = Mpad;
  p.shiftN = copies ? c.N : 0;
  p.rowmul = cs;
  p.y = y;
  p.epi_stg = (BF && env_int("SPC_PW_EPI_STG", 0) == 1 && P % 8 == 0 && !y5) ? 1 : 0;
  {
    const char* e = env_get("SPC_TILE_GROUP");
    p.tgroup = e ? atoi(e) : 1;   // measured: no effect on B200 (tools/stride_probe.py), kept as a knob
    if (p.tgroup < 1) p.tgroup = 1;
  }
  const int MBtot = Mpad / 128;
  // 3+ blocks of output channels: two groups of 256 with double-buffered accumulators (the epilogue of
  // one tile overlaps the K loop of the next) beat one group of 512 whose single accumulator set
  // serialises them, even though the activation tile is then read once per group (from L2).
  // Measured (r1, profiles/): wins for Cin <= 416 (+6..19 %), loses for Cin >= 624 where the K loop is
  // long enough to hide the epilogue and the extra activation reads cost more than the overlap gains.
  int mb = MBtot >= 3 ? (c.Cin <= 512 ? 2 : 4) : MBtot;
  // Stationary weights with several groups of output channels on 128-pixel tiles (SPC_PW_STATIONARY=1, off by default):
  // measured SLOWER than streaming them (416->416 @1024^2: 0.56 -> 0.83 ms, profiles/r2h_pw_stationary.txt) -- with
  // one block per CTA the tensor pipe issues half as many MACs per MMA slot.  The wide-N variant above is the one
  // that pays.
  {
    const char* se = env_get("SPC_PW_STATIONARY");
    const int kch = (c.Cin + BK - 1) / BK;
    p.stationary_ok = BF && ((se && atoi(se) != 0) || n256) && taps * kch * A_BLK_BYTES <= 128 * 1024;
    if (p.stationary_ok && MBtot >= 3 && !n256) mb = (taps * kch * 2 * A_BLK_BYTES <= 128 * 1024) ? 2 : 1;
    if (n256) mb = 1;
  }
  if (BF && MBtot >= 3 && !n256 && env_get("SPC_PW_MB4")) mb = 4;                 // A/B knobs
  if (BF && MBtot >= 3 && !n256 && env_get("SPC_PW_MB2")) mb = 2;
  // fp32: the 64 KB staging buffer leaves room for at most two 128-row blocks per CTA (3 stages of 48 KB)
  if (!BF && mb > 2) mb = 2;
  p.num_mg = (MBtot + mb - 1) / mb;
  p.tiles_per_image = (P + BN - 1) / BN;
  p.num_tiles = p.tiles_per_image * c.N * p.num_mg;
  if constexpr (BF) {
    if (n256) return launch_pw<T, 1, 256>(tw, tx, tx4, ty, p, st);
  }
  if (mb == 1) return launch_pw<T, 1, 128>(tw, tx, tx4, ty, p, st);
  if constexpr (BF) {
    if (mb == 2) return launch_pw<T, 2, 128>(tw, tx, tx4, ty, p, st);
    return launch_pw<T, 4, 128>(tw, tx, tx4, ty, p, st);
  } else {
    return launch_pw<T, 2, 128>(tw, tx, tx4, ty, p, st);
  }
}

// pointwise helper (1x1): Y[N][M][P] = Wp[M x Cin] * X[N][Cin][P]
template <typename T>
int run_pw(const T* w, int ld, int transpose, int M, int Cin, const T* x, const T* bias, T* y, int N, int P, void* ws,
           size_t ws_bytes, cudaStream_t st) {
  TcConv<T> c{};
  c.w = w;
  c.sm = transpose ? 1 : ld; c.sc = transpose ? ld : 1; c.flip = 0;
  c.M = M; c.Cin = Cin; c.R = 1; c.S = 1; c.ph = 0; c.pw = 0; c.H = 1; c.W = P; c.N = N; c.stride = 1;
  return run_conv_tc(c, x, bias, y, ws, ws_bytes, st);
}

// ---- wgrad kernel: dW[K x C x taps] += dY[K x P] * shift_tap(X)[C x P]^T -------------------------
// Both operands are K-major straight from NCHW (pixels = reduction dim, contiguous).  One work
// item = (group of MG 128-row blocks of dY, one block of nblk input channels, a pass of TG filter
// taps, a split of the pixel range); accumulators for all (tap, m-block) pairs of the item live in
// TMEM ((TG*MG) x nblk columns <= 512) and are flushed with fp32 atomics.
struct WgParams {
  float* dw;        // [K][C][taps] fp32 (atomic accumulation)
  int K, C, P, N;
  int nblk;         // columns (input channels) per accumulator block, multiple of 16, <= 256
  int n_blocks;     // ceil(C / nblk)
  int mgroups;      // ceil(ceil(K/128) / MG)
  int splits;       // pixel-range splits per item
  int chunks_total; // N * ceil(P/64)
  int chunks_per_image;
  int stages;
  int taps, S, ph;  // filter taps (R*S), filter width, top padding
  int TG, passes;   // taps per pass, ceil(taps / TG)
  int W, shiftN;    // OUTPUT image width; N if x is the S column-shifted copies, else 0
  int rowmul;       // input row = rowmul * output row + tap row offset
  int mrows;        // dY rows per 128-lane block (<= 128): K split EVENLY over its blocks, so every item streams the
                    // same number of valid rows and the CTAs that share an x chunk stay in lock-step (L2 hits)
  int split_major;  // 1: concurrently running CTAs cover all (m-group, channel-block, pass) groups of the SAME
                    //    pixel range, so the dY / x chunks every group re-reads come from L2, not HBM
  int pb;           // 64-pixel blocks per stage (1, or 2 = "wide" stages for 1x1 layers with multi-page channel planes)
  int dy5, x5;      // wide stages: operand moves as one 5-d box [8-ch group][px block][8 ch][128 B] (see PwParams::x5)
};

// T = float (TF32 operands): chunks of 32 pixels (one 128-byte row), 3-d boxes only (pb == 1).
template <typename T, int MG>
__global__ void __launch_bounds__(TC_THREADS, 1)
pw_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_dy, const __grid_constant__ CUtensorMap tmap_x,
                const __grid_constant__ CUtensorMap tmap_x4, const WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int b_bytes = p.nblk * 128;                        // one tap's [nblk ch][64 px] box
  const int b_slot = (b_bytes + 1023) & ~1023;
  const int stage_bytes = p.pb * (MG * A_BLK_BYTES + p.TG * b_slot);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.stages * stage_bytes);
  uint64_t* empty = full + MAX_STAGES;
  uint64_t* tfull = empty + MAX_STAGES;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tfull, 1);
    mbar_init(tempty, 128);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ngroups = p.mgroups * p.n_blocks * p.passes;
  const int num_items = ngroups * p.splits;
  const int per_split = (p.chunks_total + p.splits - 1) / p.splits;

  // item -> (split, tap pass, channel block, m group)
#define WG_DECODE(it)                                                        \
  const int sp = p.split_major ? (it) / ngroups : (it) % p.splits;           \
  const int g_ = p.split_major ? (it) % ngroups : (it) / p.splits;           \
  const int pass = g_ % p.passes;                                            \
  const int nb = (g_ / p.passes) % p.n_blocks;                               \
  const int mgp = g_ / (p.passes * p.n_blocks);                              \
  const int tap0 = pass * p.TG;                                              \
  const int ntap = min(p.TG, p.taps - tap0);                                 \
  const int c_begin = sp * per_split, c_end = min(p.chunks_total, c_begin + per_split);

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tmap_dy);
      tma_prefetch_desc(&tmap_x);
      int s = 0, ph = 0;
      for (int it = blockIdx.x; it < num_items; it += gridDim.x) {
        WG_DECODE(it)
        (void)mgp;
        for (int ch = c_begin; ch < c_end; ++ch) {
          const int n = ch / p.chunks_per_image, p0 = (ch % p.chunks_per_image) * (ROW<T> * p.pb);
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = smem + s * stage_bytes;
          mbar_arrive_expect_tx(&full[s], p.pb * (MG * p.mrows * 128 + ntap * b_bytes));
          if (p.pb == 2) {   // wide stage (taps == 1): two 64-pixel blocks of every operand row
#pragma unroll
            for (int i = 0; i < MG; ++i) {
              uint8_t* da = st + i * (2 * A_BLK_BYTES);
              const int r0 = (mgp * MG + i) * p.mrows;
              if (p.dy5) {
                tma_load_5d(da, &tmap_dy, &full[s], 0, 0, p0 >> 6, r0 >> 3, n);
              } else {
                tma_load_3d(da, &tmap_dy, &full[s], p0, r0, n);
                tma_load_3d(da + A_BLK_BYTES, &tmap_dy, &full[s], p0 + ROW<T>, r0, n);
              }
            }
            uint8_t* xa = st + MG * (2 * A_BLK_BYTES);
            if (p.x5) {
              tma_load_5d(xa, &tmap_x, &full[s], 0, 0, p0 >> 6, (nb * p.nblk) >> 3, n);
            } else {
              tma_load_3d(xa, &tmap_x, &full[s], p0, nb * p.nblk, n);
              tma_load_3d(xa + b_slot, &tmap_x, &full[s], p0 + ROW<T>, nb * p.nblk, n);
            }
            if (++s == p.stages) { s = 0; ph ^= 1; }
            continue;
          }
#pragma unroll
          for (int i = 0; i < MG; ++i)
            tma_load_3d(st + i * A_BLK_BYTES, &tmap_dy, &full[s], p0, (mgp * MG + i) * p.mrows, n);
          if (p.taps == 1) {
            tma_load_3d(st + MG * A_BLK_BYTES, &tmap_x, &full[s], p0, nb * p.nblk, n);
          } else {
            const int hq = p0 / p.W, wq = p0 - hq * p.W;
            for (int t = 0; t < ntap; ++t) {
              const int tap = tap0 + t;
              tma_load_4d(st + MG * A_BLK_BYTES + t * b_slot, &tmap_x4, &full[s], wq, hq * p.rowmul + tap / p.S - p.ph,
                          nb * p.nblk, n + (tap % p.S) * p.shiftN);
            }
          }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = Tc<T>::idesc(128, p.nblk, 0, 0);
      int s = 0, ph = 0, aph = 0;
      for (int it = blockIdx.x; it < num_items; it += gridDim.x) {
        WG_DECODE(it)
        (void)nb; (void)mgp;
        mbar_wait(tempty, aph ^ 1);
        tc_fence_after();
        for (int ch = c_begin; ch < c_end; ++ch) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * stage_bytes);
          if (p.pb == 2) {
            // wide stage: pixel block j of a 5-d box sits 1 KB after block 0 inside every 2 KB channel group; of a pair
            // of 3-d boxes, one whole box later
            const uint32_t sb = sa + MG * (2 * A_BLK_BYTES);
            const uint32_t aj = p.dy5 ? 1024 : A_BLK_BYTES, asbo = p.dy5 ? 2048 : 1024;
            const uint32_t bj = p.x5 ? 1024 : b_slot, bsbo = p.x5 ? 2048 : 1024;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t bdesc = umma_desc(sb + j * bj + ks * 32, 16, bsbo);
#pragma unroll
                for (int i = 0; i < MG; ++i) {
                  const uint64_t adesc = umma_desc(sa + i * (2 * A_BLK_BYTES) + j * aj + ks * 32, 16, asbo);
                  Tc<T>::mma(tmem_base + i * p.nblk, adesc, bdesc, idesc, (ch > c_begin || ks > 0 || j > 0) ? 1u : 0u);
                }
              }
            }
            umma_commit(&empty[s]);
            if (++s == p.stages) { s = 0; ph ^= 1; }
            continue;
          }
          const uint32_t sb = sa + MG * A_BLK_BYTES;
          for (int t = 0; t < ntap; ++t) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t bdesc = umma_desc(sb + t * b_slot + ks * 32, 16, 1024);
#pragma unroll
              for (int i = 0; i < MG; ++i) {
                const uint64_t adesc = umma_desc(sa + i * A_BLK_BYTES + ks * 32, 16, 1024);
                Tc<T>::mma(tmem_base + (t * MG + i) * p.nblk, adesc, bdesc, idesc, (ch > c_begin || ks > 0) ? 1u : 0u);
              }
            }
          }
          umma_commit(&empty[s]);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        umma_commit(tfull);
        aph ^= 1;
      }
    }
  } else {
    const int quarter = warp & 3;
    int aph = 0;
    for (int it = blockIdx.x; it < num_items; it += gridDim.x) {
      WG_DECODE(it)
      mbar_wait(tfull, aph);
      tc_fence_after();
      if (c_end > c_begin) {
#pragma unroll 1
        for (int t = 0; t < ntap; ++t) {
#pragma unroll 1
          for (int i = 0; i < MG; ++i) {
            const int rib = quarter * 32 + lane;                     // row inside the block (= TMEM lane)
            const int k = rib < p.mrows ? (mgp * MG + i) * p.mrows + rib : p.K;   // lanes >= mrows hold garbage
#pragma unroll 1
            for (int cc = 0; cc * 32 < p.nblk; ++cc) {
              uint32_t r[32];
              tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (t * MG + i) * p.nblk + cc * 32, r);
              tmem_ld_wait();
              if (k < p.K) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const int cl = cc * 32 + j;
                  const int c = nb * p.nblk + cl;
                  if (cl < p.nblk && c < p.C)
                    atomicAdd(&p.dw[((size_t)k * p.C + c) * p.taps + tap0 + t], __uint_as_float(r[j]));
                }
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(tempty);
      aph ^= 1;
    }
  }
#undef WG_DECODE
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <typename T, int MG>
int launch_wg(const CUtensorMap& tdy, const CUtensorMap& tx, const CUtensorMap& tx4, WgParams p, cudaStream_t st) {
  const int b_slot = (p.nblk * 128 + 1023) & ~1023;
  // taps per pass: TMEM columns and a stage small enough for >= 2 pipeline stages
  int TG = 512 / (MG * p.nblk);
  if (TG > p.taps) TG = p.taps;
  while (TG > 1 && MG * A_BLK_BYTES + TG * b_slot > (SMEM_LIMIT - SMEM_AUX) / 2) --TG;
  p.TG = TG;
  p.passes = (p.taps + TG - 1) / TG;
  const int stage_bytes = p.pb * (MG * A_BLK_BYTES + TG * b_slot);
  p.stages = (SMEM_LIMIT - SMEM_AUX) / stage_bytes;
  if (p.stages > 6) p.stages = 6;
  p.stages = min(p.stages, env_int("SPC_WG_STAGES", p.stages));
  SPC_REQUIRE(p.stages >= 2, "tcgen05 wgrad: smem budget");
  const int sms = sm_count();
  const int groups = p.mgroups * p.n_blocks * p.passes;
  // items = groups * splits on a persistent grid of `sms` CTAs.  Every item ends by adding its accumulators to dw with
  // fp32 atomics, and that flush is a CHIP-WIDE cost (~90 G atomics/s measured, profiles/r2_wgrad_splits.txt): with
  // few pixels per item it dominates (104->416 on a 1024x128 tile: 0.159 ms at 296 items, 0.082 at 74).  Pick the
  // split count that minimises   waves * chunks_per_item * t_chunk + items * elems_per_item / 90e9,
  // t_chunk = the slower of the item's MMA chain and its operand bytes at the per-SM share of L2 bandwidth.
  int splits = 1;
  {
    const double clk = 1.8e9;
    const double bytes_chunk = (double)p.pb * (MG * p.mrows + p.TG * p.nblk) * 128.0;
    const double mma_chunk = (double)p.pb * MG * p.TG * 4.0 * (p.nblk > 64 ? p.nblk : 64) / 256.0 * 222.0;
    const double t_chunk = (bytes_chunk / 40.0 > mma_chunk ? bytes_chunk / 40.0 : mma_chunk) / clk;
    const double elems = (double)MG * p.mrows * p.nblk * p.TG;
    const int smax = (2 * sms) / groups > 1 ? (2 * sms) / groups : 1;
    double best = 1e30;
    for (int s = smax; s >= 1; --s) {        // descending: near-ties keep the finer split (better balance)
      if (s > p.chunks_total / 8 && s > 1) continue;
      const int items_s = groups * s, waves = (items_s + sms - 1) / sms;
      const double cpi = (double)((p.chunks_total + s - 1) / s);
      const double t = waves * cpi * t_chunk + (double)items_s * elems / 90e9;
      if (t < best * 0.98) { best = t; splits = s; }
    }
  }
  if (env_get("SPC_WG_SPLIT_CEIL")) splits = (2 * sms + groups - 1) / groups;   // previous behaviour (A/B knob)
  splits = env_int("SPC_WG_SPLITS", splits);
  if (splits > p.chunks_total / 8) splits = p.chunks_total / 8;
  if (splits < 1) splits = 1;
  p.splits = splits;
  p.split_major = env_get("SPC_WG_GROUP_MAJOR") ? 0 : 1;            // A/B knob: previous item order
  const int smem = p.stages * stage_bytes + SMEM_AUX;
  auto kern = pw_wgrad_kernel<T, MG>;
  static bool attr_set = false;
  if (!attr_set) {
    SPC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set = true;
  }
  const int items = groups * p.splits;
  kern<<<items < sms ? items : sms, TC_THREADS, smem, st>>>(tdy, tx, tx4, p);
  count_launch();
  SPC_CHECK_CUDA(cudaGetLastError());
  return SPC_OK;
}

// ---- wgrad on CTA pairs (cta_group::2), 1x1 convolutions ------------------------------------------
// Default for 1x1 convolutions with >= 400 input channels (see run_wgrad; verified against the single-CTA
// kernel and against cuDNN fp32 by tests/test_gpu_fullsize_parity.py).  Why: the single-CTA kernel loads MG*128 + nblk operand rows per 64-pixel chunk for
// MG*128 x nblk accumulators (e.g. 256 + 240 rows); a pair computes M = 256*MP rows x nblk columns with each
// CTA loading only ITS 128*MP rows of dY and HALF of the nblk rows of x (256 + 120 rows for the same
// accumulators per CTA), 24-33 % fewer L2->SM bytes per MAC, and the smaller stage leaves room for 4 stages.
template <int MP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
pw_wgrad_pair_kernel(const __grid_constant__ CUtensorMap tmap_dy, const __grid_constant__ CUtensorMap tmap_x,
                     const WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int half = p.nblk / 2;                                // x rows (input channels) this CTA loads
  const int b_bytes = half * 128;
  const int b_slot = (b_bytes + 1023) & ~1023;
  const int stage_bytes = p.pb * (MP * A_BLK_BYTES + b_slot);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.stages * stage_bytes);
  uint64_t* empty = full + MAX_STAGES;
  uint64_t* tfull = empty + MAX_STAGES;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                    // 0 = leader (issues the MMAs)
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    // full: leader's arrive.expect_tx + the peer's remote arrive; empty / tfull: one multicast commit;
    // tempty (used in the leader only): the 128 epilogue threads of each CTA
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); }
    mbar_init(tfull, 1);
    mbar_init(tempty, 256);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ngroups = p.mgroups * p.n_blocks;                 // mgroups counts groups of MP row-PAIRS here
  const int num_items = ngroups * p.splits;
  const int per_split = (p.chunks_total + p.splits - 1) / p.splits;
  const uint32_t stage_tx = 2u * (uint32_t)p.pb * (uint32_t)(MP * p.mrows * 128 + b_bytes);   // both CTAs' loads land on the leader's barrier

#define WGP_DECODE(it)                                                          \
  const int sp = (it) / ngroups;                                               \
  const int g_ = (it) % ngroups;                                               \
  const int nb = g_ % p.n_blocks;                                              \
  const int mgp = g_ / p.n_blocks;                                             \
  const int c_begin = sp * per_split, c_end = min(p.chunks_total, c_begin + per_split);

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tmap_dy);
      tma_prefetch_desc(&tmap_x);
      int s = 0, ph = 0;
      for (int it = cluster_id; it < num_items; it += num_clusters) {
        WGP_DECODE(it)
        for (int ch = c_begin; ch < c_end; ++ch) {
          const int n = ch / p.chunks_per_image, p0 = (ch % p.chunks_per_image) * (64 * p.pb);
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = smem + s * stage_bytes;
          if (rank == 0) mbar_arrive_expect_tx(&full[s], stage_tx);
          else mbar_arrive_cluster(&full[s], 0);
          if (p.pb == 2) {   // wide stage: 5-d boxes [8-ch group][2 px blocks][8 ch][128 B] (see WgParams::pb)
#pragma unroll
            for (int i = 0; i < MP; ++i)
              tma_load_5d_2sm(st + i * (2 * A_BLK_BYTES), &tmap_dy, &full[s], 0, 0, p0 >> 6,
                              (((mgp * MP + i) * 2 + (int)rank) * p.mrows) >> 3, n);
            tma_load_5d_2sm(st + MP * (2 * A_BLK_BYTES), &tmap_x, &full[s], 0, 0, p0 >> 6,
                            (nb * p.nblk + (int)rank * half) >> 3, n);
            if (++s == p.stages) { s = 0; ph ^= 1; }
            continue;
          }
#pragma unroll
          for (int i = 0; i < MP; ++i)      // row pair (mgp*MP + i): this CTA's 128-lane half
            tma_load_3d_2sm(st + i * A_BLK_BYTES, &tmap_dy, &full[s], p0, ((mgp * MP + i) * 2 + (int)rank) * p.mrows, n);
          tma_load_3d_2sm(st + MP * A_BLK_BYTES, &tmap_x, &full[s], p0, nb * p.nblk + (int)rank * half, n);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = umma_idesc_bf16(256, p.nblk, 0, 0);
      int s = 0, ph = 0, aph = 0;
      for (int it = cluster_id; it < num_items; it += num_clusters) {
        WGP_DECODE(it)
        (void)nb; (void)mgp;
        mbar_wait(tempty, aph ^ 1);
        tc_fence_after();
        for (int ch = c_begin; ch < c_end; ++ch) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * stage_bytes);
          if (p.pb == 2) {
            const uint32_t sb = sa + MP * (2 * A_BLK_BYTES);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t bdesc = umma_desc(sb + j * 1024 + ks * 32, 16, 2048);
#pragma unroll
                for (int i = 0; i < MP; ++i) {
                  const uint64_t adesc = umma_desc(sa + i * (2 * A_BLK_BYTES) + j * 1024 + ks * 32, 16, 2048);
                  umma_bf16_2sm(tmem_base + i * p.nblk, adesc, bdesc, idesc, (ch > c_begin || ks > 0 || j > 0) ? 1u : 0u);
                }
              }
            }
            umma_commit_2sm(&empty[s]);
            if (++s == p.stages) { s = 0; ph ^= 1; }
            continue;
          }
          const uint32_t sb = sa + MP * A_BLK_BYTES;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t bdesc = umma_desc(sb + ks * 32, 16, 1024);
#pragma unroll
            for (int i = 0; i < MP; ++i) {
              const uint64_t adesc = umma_desc(sa + i * A_BLK_BYTES + ks * 32, 16, 1024);
              umma_bf16_2sm(tmem_base + i * p.nblk, adesc, bdesc, idesc, (ch > c_begin || ks > 0) ? 1u : 0u);
            }
          }
          umma_commit_2sm(&empty[s]);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        umma_commit_2sm(tfull);
        aph ^= 1;
      }
    }
  } else {
    const int quarter = warp & 3;
    int aph = 0;
    for (int it = cluster_id; it < num_items; it += num_clusters) {
      WGP_DECODE(it)
      mbar_wait(tfull, aph);
      tc_fence_after();
      if (c_end > c_begin) {
#pragma unroll 1
        for (int i = 0; i < MP; ++i) {
          const int rib = quarter * 32 + lane;
          const int k = rib < p.mrows ? ((mgp * MP + i) * 2 + (int)rank) * p.mrows + rib : p.K;
#pragma unroll 1
          for (int cc = 0; cc * 32 < p.nblk; ++cc) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + i * p.nblk + cc * 32, r);
            tmem_ld_wait();
            if (k < p.K) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int cl = cc * 32 + j;
                const int c = nb * p.nblk + cl;
                if (cl < p.nblk && c < p.C) atomicAdd(&p.dw[(size_t)k * p.C + c], __uint_as_float(r[j]));
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive_cluster(tempty, 0);       // both CTAs release the accumulators on the leader's barrier
      aph ^= 1;
    }
  }
#undef WGP_DECODE
  tc_fence_before();
  cluster_sync_all();                       // no CTA may exit while its peer can still signal into it
  if (warp == 1) tmem_dealloc_2sm(tmem_base, TMEM_COLS);
}

template <int MP>
int launch_wg_pair(const CUtensorMap& tdy, const CUtensorMap& tx, WgParams p, cudaStream_t st) {
  const int b_slot = ((p.nblk / 2) * 128 + 1023) & ~1023;
  const int stage_bytes = p.pb * (MP * A_BLK_BYTES + b_slot);
  p.stages = (SMEM_LIMIT - SMEM_AUX) / stage_bytes;
  if (p.stages > 6) p.stages = 6;
  p.stages = min(p.stages, env_int("SPC_WG_STAGES", p.stages));
  SPC_REQUIRE(p.stages >= 2, "tcgen05 pair wgrad: smem budget");
  const int sms = sm_count();
  const int clusters = sms / 2;
  const int groups = p.mgroups * p.n_blocks;
  int splits = 1;
  {   // same cost model as launch_wg, per CTA pair
    const double clk = 1.8e9;
    const double bytes_chunk = (double)p.pb * (MP * p.mrows + p.nblk / 2) * 128.0;          // per CTA
    const double mma_chunk = (double)p.pb * MP * 4.0 * (p.nblk > 64 ? p.nblk : 64) / 256.0 * 222.0;
    const double t_chunk = (bytes_chunk / 40.0 > mma_chunk ? bytes_chunk / 40.0 : mma_chunk) / clk;
    const double elems = 2.0 * MP * p.mrows * p.nblk;
    const int smax = (2 * clusters) / groups > 1 ? (2 * clusters) / groups : 1;
    double best = 1e30;
    for (int s = smax; s >= 1; --s) {
      if (s > p.chunks_total / 8 && s > 1) continue;
      const int items_s = groups * s, waves = (items_s + clusters - 1) / clusters;
      const double cpi = (double)((p.chunks_total + s - 1) / s);
      const double t = waves * cpi * t_chunk + (double)items_s * elems / 90e9;
      if (t < best * 0.98) { best = t; splits = s; }
    }
  }
  splits = env_int("SPC_WG_SPLITS", splits);
  if (splits > p.chunks_total / 8) splits = p.chunks_total / 8;
  if (splits < 1) splits = 1;
  p.splits = splits;
  const int smem = p.stages * stage_bytes + SMEM_AUX;
  auto kern = pw_wgrad_pair_kernel<MP>;
  static bool attr_set = false;
  if (!attr_set) {
    SPC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set = true;
  }
  const int items = groups * p.splits;
  const int grid = 2 * (items < clusters ? items : clusters);
  kern<<<grid, TC_THREADS, smem, st>>>(tdy, tx, p);
  count_launch();
  SPC_CHECK_CUDA(cudaGetLastError());
  return SPC_OK;
}

// x: activations [N][C][Hin][Wo] (taps == 1: Hin == Ho) or their S column-shifted (and, for
// stride 2, column-subsampled) copies [S][N][C][Hin][Wo].  Ho x Wo = extent of dy.
// T = float (TF32 operands): the 1-CTA kernel for every channel count, 32-pixel chunks, 3-d boxes.
template <typename T>
int run_wgrad(const T* x, const T* dy, float* dw, int K, int C, int N, int Ho, int Wo, int Hin, int R, int S, int ph,
              int stride, bool copies, cudaStream_t st) {
  constexpr bool BF = sizeof(T) == 2;
  constexpr size_t ES = sizeof(T);
  const int P = Ho * Wo;
  WgParams p{};
  p.dw = dw; p.K = K; p.C = C; p.P = P; p.N = N;
  p.taps = R * S; p.S = S; p.ph = ph; p.W = Wo; p.shiftN = copies ? N : 0; p.rowmul = stride;
  const int nblk_max = min(256, round_up(env_int("SPC_WG_NBLK", 256), 16));   // accumulator width (input channels)
  p.n_blocks = (C + nblk_max - 1) / nblk_max;
  p.nblk = round_up((C + p.n_blocks - 1) / p.n_blocks, 16);
  int MBtot = (K + 127) / 128;
  p.mrows = env_get("SPC_WG_ROWS128") ? 128 : round_up((K + MBtot - 1) / MBtot, 8);   // e.g. K = 416 -> 4 blocks of 104
  MBtot = (K + p.mrows - 1) / p.mrows;
  int MG = p.taps > 1 ? 1 : 512 / p.nblk;
  if (MG > MBtot) MG = MBtot;
  MG = min(MG, env_int("SPC_WG_MG", MG));
  MG = MG >= 4 ? 4 : (MG >= 2 ? 2 : 1);
  p.mgroups = (MBtot + MG - 1) / MG;
  p.chunks_per_image = (P + ROW<T> - 1) / ROW<T>;
  p.chunks_total = p.chunks_per_image * N;
  p.pb = 1;
  // CTA pairs (cta_group::2): measured on B200 (tools/wgrad_probe.py --pair, profiles/r2_wgrad_pair.txt): x1.11..1.32
  // for >= 416 input channels (624->416 @2048^2: 4.95 -> 3.74 ms), break-even at 416->104 / 208->52, slower for
  // the HBM-bound narrow layers (104->208: x0.75, 52->208: x0.67).  SPC_WG_2CTA=1 / SPC_WG_1CTA=1 force either.
  const bool pair = BF && p.taps == 1 && (env_get("SPC_WG_2CTA") ? true : (env_get("SPC_WG_1CTA") ? false : C >= 400)) &&
                    MBtot >= 2 && p.nblk % 16 == 0;
  // wide stages (two 64-pixel blocks per operand row and stage, 5-d boxes): for 1x1 layers whose channel planes span
  // several 2 MB pages, same reason as PwParams::x5.  SPC_WG_WIDE=0/1 overrides, SPC_WG_BOX5 (bit 0 dy, bit 1 x).
  {
    const char* we = env_get("SPC_WG_WIDE");
    const bool wide = BF && p.taps == 1 && !pair && P % 128 == 0 && (we ? atoi(we) != 0 : (size_t)P * 2 >= ((size_t)2 << 20));
    if (wide) {
      const int b_slot = (p.nblk * 128 + 1023) & ~1023;
      while (MG > 1 && 2 * 2 * (MG * A_BLK_BYTES + b_slot) > SMEM_LIMIT - SMEM_AUX) MG >>= 1;
      p.mgroups = (MBtot + MG - 1) / MG;
      p.pb = 2;
      p.chunks_per_image = P / 128;
      p.chunks_total = p.chunks_per_image * N;
      const char* be = env_get("SPC_WG_BOX5");
      const int b5 = be ? atoi(be) : 3;
      p.dy5 = ((b5 & 1) && K % 8 == 0 && p.mrows % 8 == 0) ? 1 : 0;
      p.x5 = ((b5 & 2) && C % 8 == 0 && p.nblk % 8 == 0) ? 1 : 0;
    }
  }
  CUtensorMap tdy, tx, tx4;
  int rc = p.dy5 ? make_act_tmap5(&tdy, dy, P, K, N, p.mrows / 8, 2) : make_act_tmap<T>(&tdy, dy, P, K, N, p.mrows);
  if (rc) return rc;
  if (p.taps > 1) {
    const uint64_t dims[4] = {(uint64_t)Wo, (uint64_t)Hin, (uint64_t)C, (uint64_t)N * (copies ? S : 1)};
    const uint64_t strides[4] = {0, (uint64_t)Wo * ES, (uint64_t)Hin * Wo * ES, (uint64_t)Hin * Wo * C * ES};
    const uint32_t box[4] = {(uint32_t)ROW<T>, 1, (uint32_t)p.nblk, 1};
    rc = make_tmap(&tx4, x, 4, dims, strides, box, Tc<T>::TMA_TYPE);
    if (rc) return rc;
    tx = tx4;
  } else {
    rc = p.x5 ? make_act_tmap5(&tx, x, P, C, N, p.nblk / 8, 2) : make_act_tmap<T>(&tx, x, P, C, N, p.nblk);
    if (rc) return rc;
    tx4 = tx;
  }
  if (pair) {
    // CTA pairs (see pw_wgrad_pair_kernel): row pairs of 2*mrows, MP pairs per item.  Wide stages (5-d boxes, see
    // WgParams::pb) measured x1.34..1.64 on every pair layer of the list (profiles/r2f_wgrad_pairwide.txt:
    // 1664->416 @1024^2 2.05 -> 1.53 ms = 948 TFLOP/s, 624->416 @2048^2 4.05 -> 2.54 ms); SPC_WG_PAIR_WIDE=0/1 overrides.
    const int npairs = (MBtot + 1) / 2;
    int MP = 512 / p.nblk;
    if (MP > npairs) MP = npairs;
    MP = MP >= 2 ? 2 : 1;
    CUtensorMap txh;      // x boxes of nblk/2 channels: each CTA of a pair loads its half of the block
    const char* we = env_get("SPC_WG_PAIR_WIDE");
    const bool wide = P % 128 == 0 && K % 8 == 0 && C % 8 == 0 && p.mrows % 8 == 0 && p.nblk % 16 == 0 &&
                      (we ? atoi(we) != 0 : (size_t)P * 2 >= ((size_t)2 << 20));
    if (wide) {
      const int b_slot = ((p.nblk / 2) * 128 + 1023) & ~1023;
      if (MP == 2 && env_get("SPC_WG_PAIR_MP1")) MP = 1;
      while (MP > 1 && 2 * 2 * (MP * A_BLK_BYTES + b_slot) > SMEM_LIMIT - SMEM_AUX) MP >>= 1;
      p.pb = 2;
      p.chunks_per_image = P / 128;
      p.chunks_total = p.chunks_per_image * N;
      rc = make_act_tmap5(&tdy, dy, P, K, N, p.mrows / 8, 2);
      if (rc) return rc;
      rc = make_act_tmap5(&txh, x, P, C, N, p.nblk / 16, 2);
    } else {
      rc = make_act_tmap<T>(&txh, x, P, C, N, p.nblk / 2);
    }
    if (rc) return rc;
    p.mgroups = (npairs + MP - 1) / MP;
    return MP == 2 ? launch_wg_pair<2>(tdy, txh, p, st) : launch_wg_pair<1>(tdy, txh, p, st);
  }
  if (MG == 1) return launch_wg<T, 1>(tdy, tx, tx4, p, st);
  if (MG == 2) return launch_wg<T, 2>(tdy, tx, tx4, p, st);
  return launch_wg<T, 4>(tdy, tx, tx4, p, st);
}

// ---- 3x3 stride-2 dgrad: the four output-parity classes of dX as channel groups of ONE 2x2-tap
// convolution over dY, then an interleave ("depth to space") pass.
//   dx[c, 2i+a, 2j+b] = sum_{u,v in {0,1}} sum_k Wq[(u,v)][(a,b)*C + c][k] * dy[k, i+u, j+v]
//   with Wq = w[k][c][r(a,u)][s(b,v)],  r(0,0)=1, r(1,0)=2, r(1,1)=0, r(0,1)=none (zero).
__global__ void repack_dgrad_s2_kernel(const __nv_bfloat16* __restrict__ w, __nv_bfloat16* __restrict__ wp, int K,
                                       int C, int Mpad, int Kpad) {
  const int total = 4 * Mpad * Kpad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i % Kpad;
    const int m = (i / Kpad) % Mpad;
    const int tap = i / (Kpad * Mpad);
    const int u = tap >> 1, v = tap & 1;
    __nv_bfloat16 val = __float2bfloat16(0.f);
    if (m < 4 * C && k < K) {
      const int cls = m / C, c = m % C;
      const int a = cls >> 1, b = cls & 1;
      const int r = a == 0 ? (u == 0 ? 1 : -1) : (u == 0 ? 2 : 0);
      const int sx = b == 0 ? (v == 0 ? 1 : -1) : (v == 0 ? 2 : 0);
      if (r >= 0 && sx >= 0) val = w[(((size_t)k * C + c) * 3 + r) * 3 + sx];
    }
    wp[i] = val;
  }
}
// dx[n][c][2i+a][2j+b] = t[n][(2a+b)*C + c][i][j]; 8 input pixels of both column classes per thread
__global__ void interleave_s2_kernel(const __nv_bfloat16* __restrict__ t, __nv_bfloat16* __restrict__ dx, int N, int C,
                                     int Ho, int Wo) {
  const int wv = Wo / 8;
  const size_t total = (size_t)N * C * 2 * Ho * wv;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const int oy = (int)((i / wv) % Ho);
    const int a = (int)((i / ((size_t)wv * Ho)) % 2);
    const size_t nc = i / ((size_t)wv * Ho * 2);
    const int c = (int)(nc % C);
    const size_t n = nc / C;
    const size_t plane = (size_t)Ho * Wo;
    const __nv_bfloat16* t0 = t + ((n * 4 + 2 * a) * C + c) * plane + (size_t)oy * Wo + v * 8;   // b = 0
    const uint4 e = __ldg(reinterpret_cast<const uint4*>(t0));
    const uint4 o = __ldg(reinterpret_cast<const uint4*>(t0 + (size_t)C * plane));               // b = 1
    uint4 lo, hi;
    lo.x = __byte_perm(e.x, o.x, 0x5410); lo.y = __byte_perm(e.x, o.x, 0x7632);
    lo.z = __byte_perm(e.y, o.y, 0x5410); lo.w = __byte_perm(e.y, o.y, 0x7632);
    hi.x = __byte_perm(e.z, o.z, 0x5410); hi.y = __byte_perm(e.z, o.z, 0x7632);
    hi.z = __byte_perm(e.w, o.w, 0x5410); hi.w = __byte_perm(e.w, o.w, 0x7632);
    uint4* d = reinterpret_cast<uint4*>(dx + ((nc * 2 * Ho) + 2 * oy + a) * (size_t)(2 * Wo) + v * 16);
    d[0] = lo; d[1] = hi;
  }
}

// ---- stride-2 pointwise convs: subsample / zero-upsample passes around the GEMM ------------------
// y[n,c,i,j] = x[n,c,2i,2j]; one 16-byte output vector per thread (8 bf16 / 4 fp32) from two 16-byte loads
template <typename T>
__global__ void subsample2_kernel(const T* __restrict__ x, T* __restrict__ y, size_t planes, int H, int W) {
  constexpr int V = 16 / (int)sizeof(T);
  const int Ho = H / 2, Wo = W / 2, wv = Wo / V;
  const size_t total = planes * Ho * wv;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const int oy = (int)((i / wv) % Ho);
    const size_t pl = i / ((size_t)wv * Ho);
    const uint4* src = reinterpret_cast<const uint4*>(x + (pl * H + 2 * oy) * W + v * 2 * V);
    const uint4 a = __ldg(src), b = __ldg(src + 1);
    uint4 o;
    if constexpr (sizeof(T) == 2) {
      o.x = __byte_perm(a.x, a.y, 0x5410);
      o.y = __byte_perm(a.z, a.w, 0x5410);
      o.z = __byte_perm(b.x, b.y, 0x5410);
      o.w = __byte_perm(b.z, b.w, 0x5410);
    } else {
      o.x = a.x; o.y = a.z; o.z = b.x; o.w = b.z;
    }
    *reinterpret_cast<uint4*>(y + (pl * Ho + oy) * Wo + v * V) = o;
  }
}
// dx[n,c,2i,2j] = g[n,c,i,j], zero elsewhere
template <typename T>
__global__ void upsample2_zero_kernel(const T* __restrict__ g, T* __restrict__ dx, size_t planes, int H, int W) {
  constexpr int V = 16 / (int)sizeof(T);
  const int Ho = H / 2, Wo = W / 2, wv = Wo / V;
  const size_t total = planes * Ho * wv;
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const int oy = (int)((i / wv) % Ho);
    const size_t pl = i / ((size_t)wv * Ho);
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(g + (pl * Ho + oy) * Wo + v * V));
    uint4 lo, hi;   // element e -> position 2e, zeros between
    if constexpr (sizeof(T) == 2) {
      lo.x = a.x & 0xFFFFu; lo.y = a.x >> 16; lo.z = a.y & 0xFFFFu; lo.w = a.y >> 16;
      hi.x = a.z & 0xFFFFu; hi.y = a.z >> 16; hi.z = a.w & 0xFFFFu; hi.w = a.w >> 16;
    } else {
      lo.x = a.x; lo.y = 0u; lo.z = a.y; lo.w = 0u;
      hi.x = a.z; hi.y = 0u; hi.z = a.w; hi.w = 0u;
    }
    uint4* d0 = reinterpret_cast<uint4*>(dx + (pl * H + 2 * oy) * W + v * 2 * V);
    uint4* d1 = reinterpret_cast<uint4*>(dx + (pl * H + 2 * oy + 1) * W + v * 2 * V);
    d0[0] = lo; d0[1] = hi; d1[0] = z; d1[1] = z;
  }
}
template <typename T>
int launch_resample(bool up, const void* src, void* dst, size_t planes, int H, int W, cudaStream_t st) {
  const size_t total = planes * (H / 2) * (W / 2 / (16 / sizeof(T)));
  size_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (up)
    upsample2_zero_kernel<T><<<(int)blocks, 256, 0, st>>>((const T*)src, (T*)dst, planes, H, W);
  else
    subsample2_kernel<T><<<(int)blocks, 256, 0, st>>>((const T*)src, (T*)dst, planes, H, W);
  count_launch();
  SPC_CHECK_CUDA(cudaGetLastError());
  return SPC_OK;
}

// TMA tile loads need 16-byte aligned inner coordinates (measured: tools/tma_probe.cu), so the
// horizontal taps of an R x S filter cannot be fetched as shifted boxes.  For S > 1 one pre-pass
// writes the S column-shifted, zero-filled copies  xs[s][plane][h][w] = x[plane][h][w + s - pw];
// every tap (r, s) is then an ALIGNED box of copy s at row offset r - ph.
// With column stride cs (stride-2 convs) the copies are also subsampled:
//     xs[s][plane][h][j] = x[plane][h][cs*j + s - pw],  j < W/cs.
// One 16-byte output vector (8 bf16 / 4 fp32) per thread.
template <typename T>
__global__ void shift_copies_kernel(const T* __restrict__ x, T* __restrict__ xs, size_t planes, int H, int W, int S,
                                    int pw, int cs) {
  constexpr int V = 16 / (int)sizeof(T);
  const int Wv = W / cs;
  const int wv = Wv / V;
  const size_t rows = planes * H;
  const size_t total = rows * wv * S;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const size_t row = (i / wv) % rows;
    const int sidx = (int)(i / ((size_t)wv * rows));
    const T* src = x + row * W;
    const int w0 = v * V * cs + sidx - pw;
    T e[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const int w = w0 + j * cs;
      e[j] = ((unsigned)w < (unsigned)W) ? src[w] : Tc<T>::from_float(0.f);
    }
    *reinterpret_cast<uint4*>(xs + ((size_t)sidx * rows + row) * Wv + v * V) = *reinterpret_cast<const uint4*>(e);
  }
}
// Fast path, stride 1: one thread produces the 16-byte vector (8 bf16 / 4 fp32 pixels) of ALL S copies from three
// aligned 16-byte loads (previous / own / next vector); a copy shifted by `off` columns is a 16-bit funnel shift
// (bf16) or a word selection (fp32) of that 3-vector window.  |s - pw| <= 16 B worth of pixels.
template <typename T, int S, int PW>
__global__ void __launch_bounds__(256)
shift_copies_vec_kernel(const T* __restrict__ x, T* __restrict__ xs, size_t planes, int H, int W) {
  constexpr int V = 16 / (int)sizeof(T);
  static_assert(PW <= V && S - 1 - PW <= V, "shift wider than one vector");
  const int wv = W / V;
  const size_t rows = planes * H;
  const size_t total = rows * wv;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const size_t row = i / wv;
    const uint4* src = reinterpret_cast<const uint4*>(x + row * W) + v;
    const uint4 z = make_uint4(0, 0, 0, 0);
    const uint4 a = v > 0 ? __ldg(src - 1) : z;
    const uint4 b = __ldg(src);
    const uint4 c = v < wv - 1 ? __ldg(src + 1) : z;
    const uint32_t win[13] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w, 0u};
#pragma unroll
    for (int sidx = 0; sidx < S; ++sidx) {
      const int e0 = V + sidx - PW;            // first element of the window [a|b|c]: compile-time
      uint4 o;
      if constexpr (sizeof(T) == 2) {
        const int k = e0 >> 1;
        if (e0 & 1) {
          o.x = __funnelshift_r(win[k], win[k + 1], 16);
          o.y = __funnelshift_r(win[k + 1], win[k + 2], 16);
          o.z = __funnelshift_r(win[k + 2], win[k + 3], 16);
          o.w = __funnelshift_r(win[k + 3], win[k + 4], 16);
        } else {
          o.x = win[k]; o.y = win[k + 1]; o.z = win[k + 2]; o.w = win[k + 3];
        }
      } else {
        o.x = win[e0]; o.y = win[e0 + 1]; o.z = win[e0 + 2]; o.w = win[e0 + 3];
      }
      *reinterpret_cast<uint4*>(xs + ((size_t)sidx * rows + row) * W + v * V) = o;
    }
  }
}
// Fast path, stride 2, 3 filter columns, pw = 1 (bf16): xs[s][j] = x[2j + s - 1]; 8 outputs per copy from the
// own 16 input pixels plus the last pixel of the previous vector.
__global__ void __launch_bounds__(256)
shift_copies_s2k3_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ xs, size_t planes, int H,
                         int W) {
  const int Wv = W / 2, wv = Wv / 8;
  const size_t rows = planes * H;
  const size_t total = rows * wv;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % wv);
    const size_t row = i / wv;
    const uint4* src = reinterpret_cast<const uint4*>(x + row * W) + 2 * v;
    const uint4 a = __ldg(src), b = __ldg(src + 1);
    const uint32_t prev = v > 0 ? (__ldg(reinterpret_cast<const uint32_t*>(src) - 1) >> 16) : 0u;   // x[16v - 1]
    uint4 ev, od, sh;
    ev.x = __byte_perm(a.x, a.y, 0x5410); ev.y = __byte_perm(a.z, a.w, 0x5410);     // x[16v + 0,2,4,...]
    ev.z = __byte_perm(b.x, b.y, 0x5410); ev.w = __byte_perm(b.z, b.w, 0x5410);
    od.x = __byte_perm(a.x, a.y, 0x7632); od.y = __byte_perm(a.z, a.w, 0x7632);     // x[16v + 1,3,5,...]
    od.z = __byte_perm(b.x, b.y, 0x7632); od.w = __byte_perm(b.z, b.w, 0x7632);
    sh.x = (od.x << 16) | prev;                                                      // x[16v - 1, 1, 3, ...]
    sh.y = __funnelshift_r(od.x, od.y, 16);
    sh.z = __funnelshift_r(od.y, od.z, 16);
    sh.w = __funnelshift_r(od.z, od.w, 16);
    __nv_bfloat16* dst = xs + row * Wv + v * 8;
    *reinterpret_cast<uint4*>(dst) = sh;                                  // s = 0: 2j - 1
    *reinterpret_cast<uint4*>(dst + rows * Wv) = ev;                      // s = 1: 2j
    *reinterpret_cast<uint4*>(dst + 2 * rows * Wv) = od;                  // s = 2: 2j + 1
  }
}
template <typename T>
int launch_shift_copies(const void* x, void* xs, size_t planes, int H, int W, int S, int pw, int cs, cudaStream_t st) {
  constexpr int V = 16 / (int)sizeof(T);
  const bool aligned = (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(xs) % 16 == 0);
  if (aligned && cs == 1 && W % V == 0 &&
      ((S == 7 && pw == 3) || (S == 3 && pw == 1) || (S == 5 && pw == 2) || (S == 2 && pw == 0))) {
    const size_t tot = planes * H * (W / V);
    size_t blocks = (tot + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    const T* xi = (const T*)x;
    T* xo = (T*)xs;
    if (S == 7) shift_copies_vec_kernel<T, 7, 3><<<(int)blocks, 256, 0, st>>>(xi, xo, planes, H, W);
    else if (S == 3) shift_copies_vec_kernel<T, 3, 1><<<(int)blocks, 256, 0, st>>>(xi, xo, planes, H, W);
    else if (S == 5) shift_copies_vec_kernel<T, 5, 2><<<(int)blocks, 256, 0, st>>>(xi, xo, planes, H, W);
    else shift_copies_vec_kernel<T, 2, 0><<<(int)blocks, 256, 0, st>>>(xi, xo, planes, H, W);
    count_launch();
    SPC_CHECK_CUDA(cudaGetLastError());
    return SPC_OK;
  }
  if (sizeof(T) == 2 && aligned && cs == 2 && S == 3 && pw == 1 && W % 16 == 0) {
    const size_t tot = planes * H * (W / 16);
    size_t blocks = (tot + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    shift_copies_s2k3_kernel<<<(int)blocks, 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)xs, planes, H, W);
    count_launch();
    SPC_CHECK_CUDA(cudaGetLastError());
    return SPC_OK;
  }
  const size_t total = planes * H * (W / cs / V) * S;
  size_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  shift_copies_kernel<T><<<(int)blocks, 256, 0, st>>>((const T*)x, (T*)xs, planes, H, W, S, pw, cs);
  count_launch();
  SPC_CHECK_CUDA(cudaGetLastError());
  return SPC_OK;
}

inline bool is_s2(const spc_conv_desc* d) { return d->stride_h == 2 && d->stride_w == 2; }
inline size_t align1k(size_t b) { return (b + 1023) & ~(size_t)1023; }
// fp32 storage runs on the tensor cores only when asked for TF32 (SPC_ALGO_TF32); its default is the exact direct kernel
inline bool is_tf32(const spc_conv_desc* d) { return d->dtype == SPC_F32 && d->algo == SPC_ALGO_TF32; }
inline size_t elem_bytes(const spc_conv_desc* d) { return d->dtype == SPC_BF16 ? 2 : 4; }
inline int row_elems(const spc_conv_desc* d) { return 128 / (int)elem_bytes(d); }   // channels per stage (BK)

// odd RxS "same" convs, stride 1 or 2 (TF32: stride 1 only), on 64-pixel output row segments
bool tap_shape_ok(const spc_conv_desc* d) {
  if (d->dtype != SPC_BF16 && !is_tf32(d)) return false;
  if (d->R * d->S == 1 || d->R * d->S > 49) return false;
  if ((d->R & 1) == 0 || (d->S & 1) == 0) return false;
  const bool s1 = d->stride_h == 1 && d->stride_w == 1, s2 = d->stride_h == 2 && d->stride_w == 2;
  if (!s1 && !s2) return false;
  if (s2 && (d->H % 2 || d->W % 2)) return false;
  if (s2 && is_tf32(d)) return false;   // 3x3 stride 2 in fp32 stays on the direct kernel
  const int Wo = d->W / d->stride_w;
  if (Wo % 64 != 0) return false;
  return (long long)d->H * d->W < (1ll << 31);
}

bool pw_shape_ok(const spc_conv_desc* d) {
  if (d->dtype != SPC_BF16 && !is_tf32(d)) return false;
  if (d->R != 1 || d->S != 1) return false;
  long long P = (long long)d->H * d->W;
  if (is_s2(d)) {
    if (d->H % 2 || d->W % 32) return false;   // 16-byte vectors on both sides of the resample
    P /= 4;
  } else if (d->stride_h != 1 || d->stride_w != 1) {
    return false;
  }
  // TMA strides are multiples of 16 bytes: P % 8 (bf16) / P % 4 (fp32)
  if (P % (16 / (long long)elem_bytes(d)) != 0 || P >= (1ll << 31)) return false;
  return true;
}

}  // namespace

bool tc_supported(const spc_conv_desc* d, int op) {
  if (pw_shape_ok(d)) return true;
  if (tap_shape_ok(d)) {
    if (tc_workspace_bytes(d, op) > (24ull << 30)) return false;   // shifted copies would not fit comfortably
    if (op == 1 && is_s2(d)) return d->R == 3 && d->S == 3 && 4 * d->C <= 2048;   // parity-class dgrad
    return true;
  }
  return false;
}

// workspace = [repacked weights | subsampled activations (stride-2 only)]
static size_t wbytes(const spc_conv_desc* d, int op) {
  const size_t taps = (size_t)d->R * d->S, es = elem_bytes(d);
  const int bk = row_elems(d);
  if (op == 0) return align1k(taps * round_up(d->K, 128) * round_up(d->C, bk) * es + 1024);
  if (op == 1) return align1k(taps * round_up(d->C, 128) * round_up(d->K, bk) * es + 1024);
  return 0;
}
size_t tc_workspace_bytes(const spc_conv_desc* d, int op) {
  const size_t taps = (size_t)d->R * d->S, es = elem_bytes(d);
  const int cs = d->stride_w;
  const bool bf = d->dtype == SPC_BF16;
  size_t b = wbytes(d, op) + 4096;
  if (taps == 1) {
    if (is_s2(d)) b += align1k((size_t)d->N * d->C * (d->H / 2) * (d->W / 2) * es) + 1024;
    return b;
  }
  const size_t Ho = d->H / cs, Wo = d->W / cs;
  if (op == 1 && is_s2(d)) {
    // Wq[4][4C pad][K pad] + 2 column-shifted copies of dy + the 4-class output planes
    b = align1k(4ull * round_up(4 * d->C, 128) * round_up(d->K, BK) * 2) + 4096;
    b += align1k(2ull * d->N * d->K * Ho * Wo * 2) + align1k(4ull * d->N * d->C * Ho * Wo * 2) + 4096;
    return b;
  }
  if (bf && op != 2 && !env_get("SPC_TAP_V1") &&
      tap_v2_supported(op == 1 ? d->C : d->K, op == 1 ? d->K : d->C, d->R, d->S, d->H, d->W, d->N, cs))
    return b;               // conv_tap.cu forms the horizontal taps in shared memory: no copies
  if (bf && op == 2 && !env_get("SPC_TAP_V1") && wgrad_tap_supported(d->K, d->C, d->R, d->S, d->H, d->W, cs))
    return b;               // wgrad_tap.cu likewise
  if (d->S > 1 || cs > 1)   // S column-shifted (stride 2: also subsampled) copies of the conv input
    b += align1k((size_t)d->S * d->N * (op == 1 ? d->K : d->C) * d->H * Wo * es) + 2048;
  return b;
}

namespace {

template <typename T>
int conv_fwd_t(const spc_conv_desc* d, const T* x, const T* w, const T* bias, T* y, void* ws, size_t ws_bytes,
               cudaStream_t st) {
  if (d->R * d->S > 1) {
    TcConv<T> c{};
    c.w = w;
    c.sm = (long long)d->C * d->R * d->S; c.sc = (long long)d->R * d->S; c.flip = 0;
    c.M = d->K; c.Cin = d->C; c.R = d->R; c.S = d->S; c.ph = d->pad_h; c.pw = d->pad_w;
    c.H = d->H; c.W = d->W; c.N = d->N; c.stride = d->stride_h;
    return run_conv_tc(c, x, bias, y, ws, ws_bytes, st);
  }
  if (is_s2(d)) {   // Y = W * subsample(X)
    T* xs = reinterpret_cast<T*>(align1k(reinterpret_cast<uintptr_t>(ws) + wbytes(d, 0)));
    int rc = launch_resample<T>(false, x, xs, (size_t)d->N * d->C, d->H, d->W, st);
    if (rc) return rc;
    return run_pw(w, d->C, 0, d->K, d->C, xs, bias, y, d->N, (d->H / 2) * (d->W / 2), ws, wbytes(d, 0), st);
  }
  return run_pw(w, d->C, 0, d->K, d->C, x, bias, y, d->N, d->H * d->W, ws, ws_bytes, st);
}

// every dgrad except 3x3 stride 2 (bf16 only, tc_conv_dgrad)
template <typename T>
int conv_dgrad_t(const spc_conv_desc* d, const T* dy, const T* w, T* dx, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (d->R * d->S > 1) {   // stride-1 dgrad = correlation of dY with the transposed, 180-degree rotated filter
    TcConv<T> c{};
    c.w = w;
    c.sm = (long long)d->R * d->S; c.sc = (long long)d->C * d->R * d->S; c.flip = 1;
    c.M = d->C; c.Cin = d->K; c.R = d->R; c.S = d->S; c.ph = d->R - 1 - d->pad_h; c.pw = d->S - 1 - d->pad_w;
    c.H = d->H; c.W = d->W; c.N = d->N; c.stride = 1;
    return run_conv_tc(c, dy, (const T*)nullptr, dx, ws, ws_bytes, st);
  }
  if (is_s2(d)) {   // dX = zero_upsample(W^T * dY)
    T* gs = reinterpret_cast<T*>(align1k(reinterpret_cast<uintptr_t>(ws) + wbytes(d, 1)));
    int rc = run_pw(w, d->C, 1, d->C, d->K, dy, (const T*)nullptr, gs, d->N, (d->H / 2) * (d->W / 2), ws, wbytes(d, 1), st);
    if (rc) return rc;
    return launch_resample<T>(true, gs, dx, (size_t)d->N * d->C, d->H, d->W, st);
  }
  return run_pw(w, d->C, 1, d->C, d->K, dy, (const T*)nullptr, dx, d->N, d->H * d->W, ws, ws_bytes, st);
}

template <typename T>
int conv_wgrad_t(const spc_conv_desc* d, const T* x, const T* dy, float* dw, void* ws, size_t ws_bytes,
                 cudaStream_t st) {
  if (d->R * d->S > 1) {
    const int cs = d->stride_h;
    if constexpr (sizeof(T) == 2) {
      if (!env_get("SPC_TAP_V1") && wgrad_tap_supported(d->K, d->C, d->R, d->S, d->H, d->W, cs))
        return run_wgrad_tap(x, dy, dw, d->K, d->C, d->N, d->H, d->W, d->R, d->S, st);
    }
    const bool copies = d->S > 1 || cs > 1;
    if (copies) {
      SPC_REQUIRE(ws && ws_bytes >= tc_workspace_bytes(d, 2), "tcgen05 wgrad: workspace too small");
      void* xs = reinterpret_cast<void*>(align1k(reinterpret_cast<uintptr_t>(ws)));
      int rc = launch_shift_copies<T>(x, xs, (size_t)d->N * d->C, d->H, d->W, d->S, d->pad_w, cs, st);
      if (rc) return rc;
      x = reinterpret_cast<const T*>(xs);
    }
    return run_wgrad(x, dy, dw, d->K, d->C, d->N, d->H / cs, d->W / cs, d->H, d->R, d->S, d->pad_h, cs, copies, st);
  }
  if (is_s2(d)) {
    SPC_REQUIRE(ws && ws_bytes >= tc_workspace_bytes(d, 2), "tcgen05 wgrad: workspace too small");
    T* xs = reinterpret_cast<T*>(align1k(reinterpret_cast<uintptr_t>(ws)));
    int rc = launch_resample<T>(false, x, xs, (size_t)d->N * d->C, d->H, d->W, st);
    if (rc) return rc;
    return run_wgrad<T>(xs, dy, dw, d->K, d->C, d->N, 1, (d->H / 2) * (d->W / 2), 1, 1, 1, 0, 1, false, st);
  }
  return run_wgrad(x, dy, dw, d->K, d->C, d->N, 1, d->H * d->W, 1, 1, 1, 0, 1, false, st);
}

}  // namespace

int tc_conv_fwd(const spc_conv_desc* d, const void* x, const void* w, const void* bias, void* y, void* ws,
                size_t ws_bytes, cudaStream_t st) {
  SPC_REQUIRE(ws && ws_bytes >= tc_workspace_bytes(d, 0), "tcgen05 conv: workspace too small");
  if (d->dtype == SPC_F32)
    return conv_fwd_t(d, (const float*)x, (const float*)w, (const float*)bias, (float*)y, ws, ws_bytes, st);
  return conv_fwd_t(d, (const __nv_bfloat16*)x, (const __nv_bfloat16*)w, (const __nv_bfloat16*)bias,
                    (__nv_bfloat16*)y, ws, ws_bytes, st);
}

int tc_conv_dgrad(const spc_conv_desc* d, const void* dy, const void* w, void* dx, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
  // dX[C x P] = W^T[C x K] * dY[K x P]
  SPC_REQUIRE(ws && ws_bytes >= tc_workspace_bytes(d, 1), "tcgen05 conv: workspace too small");
  if (d->dtype == SPC_F32) return conv_dgrad_t(d, (const float*)dy, (const float*)w, (float*)dx, ws, ws_bytes, st);
  if (d->R * d->S > 1 && is_s2(d)) {   // 3x3 stride 2: four parity classes as channel groups, then interleave
    const int Ho = d->H / 2, Wo = d->W / 2;
    const int Mq = 4 * d->C, Mpad = round_up(Mq, 128), Kpad = round_up(d->K, BK);
    uintptr_t a = align1k(reinterpret_cast<uintptr_t>(ws));
    __nv_bfloat16* wq = reinterpret_cast<__nv_bfloat16*>(a);
    a = align1k(a + (size_t)4 * Mpad * Kpad * 2);
    __nv_bfloat16* tmp = reinterpret_cast<__nv_bfloat16*>(a);
    a = align1k(a + (size_t)4 * d->N * d->C * Ho * Wo * 2);
    {
      const int total = 4 * Mpad * Kpad;
      int blocks = (total + 255) / 256;
      if (blocks > 1184) blocks = 1184;
      repack_dgrad_s2_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(w), wq, d->K, d->C, Mpad, Kpad);
      count_launch();
      SPC_CHECK_CUDA(cudaGetLastError());
    }
    TcConv<__nv_bfloat16> c{};
    c.prepacked = wq;
    c.M = Mq; c.Cin = d->K; c.R = 2; c.S = 2; c.ph = 0; c.pw = 0; c.H = Ho; c.W = Wo; c.N = d->N; c.stride = 1;
    int rc = run_conv_tc(c, reinterpret_cast<const __nv_bfloat16*>(dy), (const __nv_bfloat16*)nullptr, tmp, reinterpret_cast<void*>(a),
                         ws_bytes - (a - reinterpret_cast<uintptr_t>(ws)), st);
    if (rc) return rc;
    const size_t total = (size_t)d->N * d->C * 2 * Ho * (Wo / 8);
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    interleave_s2_kernel<<<(int)blocks, 256, 0, st>>>(tmp, reinterpret_cast<__nv_bfloat16*>(dx), d->N, d->C, Ho, Wo);
    count_launch();
    SPC_CHECK_CUDA(cudaGetLastError());
    return SPC_OK;
  }
  return conv_dgrad_t(d, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)w, (__nv_bfloat16*)dx, ws, ws_bytes, st);
}

int tc_conv_wgrad(const spc_conv_desc* d, const void* x, const void* dy, float* dw, int accumulate, void* ws,
                  size_t ws_bytes, cudaStream_t st) {
  // the kernel accumulates with atomics; api.cu has already zeroed dw when !accumulate
  (void)accumulate;
  if (d->dtype == SPC_F32) return conv_wgrad_t(d, (const float*)x, (const float*)dy, dw, ws, ws_bytes, st);
  return conv_wgrad_t(d, (const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, dw, ws, ws_bytes, st);
}

// Y[M][P] = W[M][Cin] * X[Cin][P] (bf16; w row-major with leading dimension ld) and dW[K][C] += dY[K][P] * X[C][P]^T on
// the pointwise tcgen05 kernels -- used by the halo fix-up (api.cu), where "channels" are (c, r, s) triples of the
// filter and "pixels" are the boundary outputs
size_t tc_pw_workspace_bytes(int M, int Cin) { return (size_t)round_up(M, 128) * round_up(Cin, BK) * 2 + 4096; }
int tc_pw_fwd(const void* w, int ld, int M, int Cin, const void* x, const void* bias, void* y, int P, void* ws, size_t ws_bytes,
              cudaStream_t st) {
  return run_pw(reinterpret_cast<const __nv_bfloat16*>(w), ld, 0, M, Cin, reinterpret_cast<const __nv_bfloat16*>(x),
                reinterpret_cast<const __nv_bfloat16*>(bias), reinterpret_cast<__nv_bfloat16*>(y), 1, P, ws, ws_bytes, st);
}
int tc_pw_wgrad(const void* x, const void* dy, float* dw, int K, int C, int P, cudaStream_t st) {
  return run_wgrad(reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<const __nv_bfloat16*>(dy), dw, K, C, 1, 1, P, 1, 1, 1,
                   0, 1, false, st);
}

int make_tmap_ex(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                 const uint32_t* box, int swizzle128) {
  return make_tmap_sw(m, base, rank, dims, strides_bytes, box,
                      swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE);
}
int tc_sm_count() { return sm_count(); }

}  // namespace spc

// tuning probes (tools/wgrad_probe.py) change SPC_* knobs inside one process: forget the cached values
extern "C" void spc_reload_env(void) { spc::g_env_n = 0; }
