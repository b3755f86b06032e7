// Dev probe: can fp32 activations in NCHW feed a tcgen05 kind::tf32 MMA as they are?  One 128 x 128 x 32 tile, fed by
// TMA the way gemm_tc.cu feeds its bf16 operands (one 128-byte swizzle row = 32 fp32 channels or pixels).
// A = W[128 m][32 k] is K-major in every mode.  B = X:
//   mode 0: MN-major [32 k][128 px] (pixels contiguous), 4 blocks of [32 k][32 px], TMA SWIZZLE_128B, descriptor layout 2,
//           LBO = 4 KB (next 32-pixel block), SBO = 1 KB.  This is the bf16 kernels' descriptor one-to-one and is NOT
//           expected to work for 32-bit elements: a 16-byte swizzle chunk holds only 4 fp32 values, while an MN-major
//           TF32 operand is swizzled in 32-byte atoms (the reason the 32-byte-atom layout exists).
//   mode 1: K-major [128 px][32 k] (the wgrad form), SWIZZLE_128B.
//   modes 2-5: MN-major as mode 0, loaded with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B and described with descriptor layout 1
//           (128-byte swizzle, 32-byte atoms) and the (LBO, SBO) pairs of the table in main().  With 4 atoms of 32 B per
//           128-byte row the pattern repeats every 4 rows, so one K = 8 MMA spans two 4-row K groups 512 B apart: mode 4
//           (LBO = 4 KB, SBO = 512 B) is the natural candidate, mode 5 the swap.
// The 32-byte-atom tile TMA writes is also dumped (x[k][px] = k * 128 + px) to show its pattern.
// Compared on the host with a double-precision product of the same inputs.  Two input sets: TF32-representable values
// (every product and partial sum is exact in fp32, so the result must match exactly) and random fp32 values (reports the
// error against the exact product and against products of TF32-truncated operands).
// Measured on B200 (profiles/r3_tf32_mma_probe.txt): modes 1 and 4 are exact; gemm_tc.cu uses mode 4 for fp32.
//   nvcc -gencode arch=compute_100a,code=sm_100a -o tf32_mma_probe tools/tf32_mma_probe.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../mpi4dl_b200/csrc/tc_common.cuh"
using namespace spc::tc;

struct Mode {
  const char* name;
  int b_kmajor;                 // 1: B stored [px][k] (K-major), 0: [k][px] (MN-major)
  CUtensorMapSwizzle swz;       // TMA swizzle of B
  uint32_t layout, lbo, sbo;    // B descriptor
};

__global__ void probe(const __grid_constant__ CUtensorMap ta, const __grid_constant__ CUtensorMap tb, Mode md, float* d,
                      float* sdump) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sa = sm;                 // 16 KB
  uint8_t* sb = sm + 16384;         // 16 KB
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm + 32768);
  uint64_t* mbar = bar + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_init(mbar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(bar, 32768);
    tma_load_2d(sa, &ta, bar, 0, 0);
    if (!md.b_kmajor)
      for (int j = 0; j < 4; ++j) tma_load_2d(sb + j * 4096, &tb, bar, j * 32, 0);
    else
      tma_load_2d(sb, &tb, bar, 0, 0);
    mbar_wait(bar, 0);
    tc_fence_after();
    const uint32_t idesc = umma_idesc_tf32(128, 128, 0, md.b_kmajor ? 0 : 1);
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t adesc = umma_desc(smem_u32(sa) + ks * 32, 16, 1024);
      // k-step of 8: K-major +32 B along the row, MN-major +8 rows of 128 B
      const uint64_t bdesc = umma_desc(smem_u32(sb) + (md.b_kmajor ? ks * 32 : ks * 1024), md.lbo, md.sbo, md.layout);
      umma_tf32(tmem, adesc, bdesc, idesc, ks ? 1u : 0u);
    }
    umma_commit(mbar);
  }
  __syncwarp();
  mbar_wait(bar, 0);
  if (sdump)
    for (int i = threadIdx.x; i < 4096; i += blockDim.x) sdump[i] = reinterpret_cast<const float*>(sb)[i];
  mbar_wait(mbar, 0);
  tc_fence_after();
  for (int cc = 0; cc < 4; ++cc) {
    uint32_t r[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + cc * 32, r);
    tmem_ld_wait();
    for (int j = 0; j < 32; ++j) d[(warp * 32 + lane) * 128 + cc * 32 + j] = __uint_as_float(r[j]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

typedef CUresult (*Enc)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static float trunc_tf32(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  u &= 0xFFFFE000u;
  memcpy(&v, &u, 4);
  return v;
}

static int make2d(Enc enc, CUtensorMap* m, void* base, int inner, int outer, int box_inner, int box_outer,
                  CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  cuuint64_t gd[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t gs[1] = {(cuuint64_t)inner * 4};
  cuuint32_t bx[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer}, es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { printf("encode failed %d\n", (int)r); return 1; }
  return 0;
}

int main() {
  void* fp = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q) != cudaSuccess || !fp) {
    printf("no cuTensorMapEncodeTiled\n");
    return 1;
  }
  Enc enc = (Enc)fp;
  const int M = 128, N = 128, K = 32;
  float *hw = (float*)malloc(M * K * 4), *hx = (float*)malloc(K * N * 4), *hd = (float*)malloc(M * N * 4);
  float *dw, *dx, *dd;
  cudaMalloc(&dw, M * K * 4); cudaMalloc(&dx, K * N * 4); cudaMalloc(&dd, M * N * 4);
  cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 40 * 1024);
  const Mode modes[] = {
      {"MN-major SW128 (bf16 descriptor)  LBO 4096 SBO 1024", 0, CU_TENSOR_MAP_SWIZZLE_128B, 2, 4096, 1024},
      {"K-major  SW128                    LBO   16 SBO 1024", 1, CU_TENSOR_MAP_SWIZZLE_128B, 2, 16, 1024},
      {"MN-major SW128 32B atoms          LBO 4096 SBO 1024", 0, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, UMMA_SW128_ATOM32, 4096, 1024},
      {"MN-major SW128 32B atoms          LBO 1024 SBO 4096", 0, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, UMMA_SW128_ATOM32, 1024, 4096},
      {"MN-major SW128 32B atoms          LBO 4096 SBO  512", 0, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, UMMA_SW128_ATOM32, 4096, 512},
      {"MN-major SW128 32B atoms          LBO  512 SBO 4096", 0, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, UMMA_SW128_ATOM32, 512, 4096},
  };
  const int NM = sizeof(modes) / sizeof(modes[0]);
  int ok_mode[8] = {0};
  float* ddump;
  cudaMalloc(&ddump, 4096 * 4);
  srand(1234);
  for (int set = 0; set < 3; ++set) {
    // set 0: TF32-representable values, set 1: random fp32, set 2: x = k * 128 + px (smem dump of the 32-byte-atom tile)
    for (int i = 0; i < M * K; ++i)
      hw[i] = set == 0 ? (float)(rand() % 257 - 128) / 64.f : (float)rand() / RAND_MAX * 2.f - 1.f;
    for (int i = 0; i < K * N; ++i)
      hx[i] = set == 0 ? (float)(rand() % 257 - 128) / 64.f : set == 1 ? (float)rand() / RAND_MAX * 2.f - 1.f : (float)i;
    for (int mode = 0; mode < NM; ++mode) {
      const Mode& md = modes[mode];
      if (set == 2 && mode != 4) continue;
      float* hxs = (float*)malloc(K * N * 4);
      for (int k = 0; k < K; ++k)
        for (int n = 0; n < N; ++n) hxs[md.b_kmajor ? n * K + k : k * N + n] = hx[k * N + n];
      cudaMemcpy(dw, hw, M * K * 4, cudaMemcpyHostToDevice);
      cudaMemcpy(dx, hxs, K * N * 4, cudaMemcpyHostToDevice);
      cudaMemset(dd, 0, M * N * 4);
      CUtensorMap ta, tb;
      if (make2d(enc, &ta, dw, K, M, 32, 128)) return 1;
      if (md.b_kmajor ? make2d(enc, &tb, dx, K, N, 32, 128) : make2d(enc, &tb, dx, N, K, 32, 32, md.swz)) return 1;
      probe<<<1, 128, 40 * 1024>>>(ta, tb, md, dd, set == 2 ? ddump : nullptr);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("mode %d set %d: launch failed: %s\n", mode, set, cudaGetErrorString(e)); return 1; }
      free(hxs);
      if (set == 2) {
        // smem row r (128 B) of pixel block 0 = channel r; print which pixels each of its four 32-byte slots holds
        float hs[4096];
        cudaMemcpy(hs, ddump, sizeof(hs), cudaMemcpyDeviceToHost);
        printf("32-byte-atom tile written by TMA, pixel block 0: row r, slot j -> (channel, first pixel) of the 8 values\n");
        for (int r = 0; r < 8; ++r) {
          printf("  row %d:", r);
          for (int j = 0; j < 4; ++j) {
            const int v = (int)hs[r * 32 + j * 8];
            bool run = true;
            for (int t = 1; t < 8; ++t) run &= (int)hs[r * 32 + j * 8 + t] == v + t;
            printf("  (%2d,%3d)%s", v / 128, v % 128, run ? "" : "*");
          }
          printf("\n");
        }
        continue;
      }
      cudaMemcpy(hd, dd, M * N * 4, cudaMemcpyDeviceToHost);
      double max_exact = 0, max_trunc = 0, scale = 0;
      for (int m = 0; m < M; ++m)
        for (int n = 0; n < N; ++n) {
          double s = 0, st = 0;
          for (int k = 0; k < K; ++k) {
            s += (double)hw[m * K + k] * hx[k * N + n];
            st += (double)trunc_tf32(hw[m * K + k]) * trunc_tf32(hx[k * N + n]);
          }
          const double g = hd[m * N + n];
          max_exact = fmax(max_exact, fabs(g - s));
          max_trunc = fmax(max_trunc, fabs(g - st));
          scale = fmax(scale, fabs(s));
        }
      const bool ok = set == 0 ? max_exact == 0.0 : max_trunc <= 1e-5 * scale;
      ok_mode[mode] += ok;
      printf("mode %d %s, %s: max |err| vs exact %.3g, vs truncated-TF32 operands %.3g (|ref| max %.3g)  %s\n", mode,
             md.name, set == 0 ? "TF32-representable" : "random fp32       ", max_exact, max_trunc, scale,
             ok ? "OK" : "FAIL");
    }
  }
  int mn_ok = 0;
  for (int mode = 2; mode < NM; ++mode) mn_ok |= ok_mode[mode] == 2;
  const int bad = ok_mode[1] != 2 || !mn_ok;
  printf("K-major TF32: %s;  MN-major TF32 (32-byte atoms):", ok_mode[1] == 2 ? "OK" : "FAILED");
  for (int mode = 2; mode < NM; ++mode)
    if (ok_mode[mode] == 2) printf(" mode %d OK", mode);
  printf("%s\n", mn_ok ? "" : " no layout tried works");
  printf(bad ? "TF32 PROBE FAILED\n" : "TF32 PROBE OK\n");
  return bad ? 1 : 0;
}
