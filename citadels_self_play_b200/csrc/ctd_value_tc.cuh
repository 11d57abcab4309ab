// ctd_value_tc.cuh -- the value model's dense layers on the 5th-generation tensor cores (tcgen05 + TMEM).
//
//   Y[M x N] = act( X[M x K] . W[N x K]^T + b )      fp32 in / fp32 out
//
// The reference evaluates ValueOnlyNN in fp32 (algorithms/models.py:17-23) and parity is asked to 1e-5 relative.
// A single TF32 pass (10-bit mantissa) is ~1e-3, the usual two-term split (3xTF32) measured 1-3e-5 on this model,
// so each fp32 operand is split into THREE TF32 terms, x = x0 + x1 + x2 (x0 = rna(x), x1 = rna(x - x0),
// x2 = rna(x - x0 - x1): 33 mantissa bits, i.e. exact), and the six products of weight >= 2^-22,
//   x0.w0 + x0.w1 + x1.w0 + x0.w2 + x1.w1 + x2.w0,
// are accumulated in fp32 in TMEM.  The layers are tiny (757 kFLOP per leaf), so six passes cost nothing.
// Measured on B200 (profiles/r01_value_tc_accuracy.md): with the operands represented exactly the remaining error comes
// from the accumulator update -- every instruction rounds (toward zero, it seems: the error is a bias) once when it adds
// its eight products to the fp32 accumulator in TMEM, at the accumulator's magnitude.  Padding instructions with zeros
// (twice the instructions) doubles the error; dealing the K slices over FOUR accumulators (all 512 TMEM columns), each a
// quarter of the magnitude, and summing them in fp32 registers in the epilogue divides it by four: 1.0e-5 max / 1.2e-6 mean
// absolute on outputs of scale 5, and deep-MCCFR trees within 3.3e-6 of the reference's (the fp32 CUDA-core kernel
// ctd_k_value_mlp: 3.2e-6), against 1.3e-5 with one accumulator.  ctd_set_value_backend selects the fp32 kernel.
//
// One CTA (128 threads) computes a 128 x 128 output tile:
//   * all four warps stream K in slices of 32 floats: 16-byte global loads, split into hi/lo, st.shared into the
//     canonical K-major no-swizzle UMMA layout (8-row x 16-byte core matrices; K-adjacent cores LBO = 128 B apart,
//     8-row groups SBO = 1024 B apart), two stages so the loads of slice s+1 overlap the MMAs of slice s;
//   * one elected thread issues tcgen05.mma.cta_group::1.kind::tf32 (M = 128, N = 128, K = 8 per instruction)
//     and tcgen05.commit's to the stage's mbarrier, which is what frees the stage for the next load;
//   * four accumulators (128 lanes x 128 columns fp32 each) live in TMEM, K slice kk of every stage goes to accumulator kk;
//     the epilogue reads them back with tcgen05.ld.32x32b (each warp its own 32 lanes, one row per thread), sums them,
//     adds the bias, applies ReLU and stores.
// Weights total 1.5 MB and stay L2-resident; activations between layers round-trip through L2 (M x 512 floats).
#pragma once
#include <stdint.h>
#include <cuda.h>   // CUtensorMap (the descriptor type only; the encoder is fetched from the driver at run time)

#define CTD_TC_BM 128
#define CTD_TC_BN 128
#define CTD_TC_BK 32
#define CTD_TC_TERMS 3
#define CTD_TC_TILE_BYTES (128 * CTD_TC_BK * 4)                   /* 16 KB: one operand tile, one split term */
#define CTD_TC_STAGE_BYTES (2 * CTD_TC_TERMS * CTD_TC_TILE_BYTES) /* A0 A1 A2 B0 B1 B2 */
#define CTD_TC_ACCS 4 /* TMEM accumulators the K slices are dealt over (each rounds once per instruction at its own, smaller, magnitude); summed in fp32 registers in the epilogue */
#define CTD_TC_SMEM (2 * CTD_TC_STAGE_BYTES + 1024)               /* two stages + alignment slack */
#define CTD_TC_SPIN_LIMIT (1u << 24)

__device__ __forceinline__ uint32_t ctd_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ctd_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ctd_smem_u32(bar)), "r"(count));
}
// bounded wait: a barrier that never flips sets *err instead of hanging the GPU
__device__ __forceinline__ bool ctd_mbar_wait(uint64_t* bar, uint32_t parity, int* err) {
  const uint32_t addr = ctd_smem_u32(bar);
  for (uint32_t spin = 0; spin < CTD_TC_SPIN_LIMIT; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return true;
  }
  if (err) atomicExch(err, 1);
  return false;
}

__device__ __forceinline__ float ctd_to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// K-major, no swizzle: start address, LBO (K-adjacent core matrices), SBO (8-row groups), descriptor version 1
__device__ __forceinline__ uint64_t ctd_umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// kind::tf32, fp32 accumulate, A and B K-major, M = 128, N = 128
#define CTD_TC_IDESC ((1u << 4) | (2u << 7) | (2u << 10) | ((CTD_TC_BN >> 3) << 17) | ((CTD_TC_BM >> 4) << 24))

__device__ __forceinline__ void ctd_umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"((uint32_t)CTD_TC_IDESC), "r"(accumulate)
      : "memory");
}

// one 16-byte chunk of an operand tile: split into three TF32 terms and store them in the UMMA layout
// (term t of the operand lives at tile + t * CTD_TC_TILE_BYTES)
__device__ __forceinline__ void ctd_tc_split3(float x, float& t0, float& t1, float& t2) {
  t0 = ctd_to_tf32(x);
  const float r1 = x - t0;  // exact
  t1 = ctd_to_tf32(r1);
  t2 = ctd_to_tf32(r1 - t1);
}
__device__ __forceinline__ void ctd_tc_stage_chunk(uint8_t* tile, int row, int chunk, float4 v) {
  float4 a, b, c;
  ctd_tc_split3(v.x, a.x, b.x, c.x);
  ctd_tc_split3(v.y, a.y, b.y, c.y);
  ctd_tc_split3(v.z, a.z, b.z, c.z);
  ctd_tc_split3(v.w, a.w, b.w, c.w);
  const int off = (row >> 3) * 1024 + chunk * 128 + (row & 7) * 16;
  *reinterpret_cast<float4*>(tile + off) = a;
  *reinterpret_cast<float4*>(tile + CTD_TC_TILE_BYTES + off) = b;
  *reinterpret_cast<float4*>(tile + 2 * CTD_TC_TILE_BYTES + off) = c;
}

__global__ void __launch_bounds__(128) ctd_k_linear_tc(const float* __restrict__ X, int ldx, const float* __restrict__ W, int ldw,
                                                       const float* __restrict__ bias, float* __restrict__ Y, int ldy, int M, int K,
                                                       int relu, int* err) {
  extern __shared__ uint8_t tc_smem_raw[];
  __shared__ uint64_t bars[2];
  __shared__ uint32_t tmem_base_slot;
  uint8_t* smem = (uint8_t*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int m0 = blockIdx.x * CTD_TC_BM, n0 = blockIdx.y * CTD_TC_BN;

  if (warp == 0) {  // TMEM: 128 columns for the fp32 accumulator tile
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(ctd_smem_u32(&tmem_base_slot)), "r"((uint32_t)(128 * CTD_TC_ACCS)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    ctd_mbar_init(&bars[0], 1);
    ctd_mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = tmem_base_slot;

  const int stages = K / CTD_TC_BK;
  bool ok = true;
  for (int s = 0; s < stages; ++s) {
    const int buf = s & 1;
    uint8_t* st = smem + buf * CTD_TC_STAGE_BYTES;
    if (s >= 2) ok = ctd_mbar_wait(&bars[buf], (uint32_t)(((s >> 1) - 1) & 1), err) && ok;  // MMAs of slice s-2 are done
    const int k0 = s * CTD_TC_BK;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + 128 * i, row = idx >> 3, chunk = idx & 7;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + row < M) a = *reinterpret_cast<const float4*>(X + (size_t)(m0 + row) * ldx + k0 + 4 * chunk);
      ctd_tc_stage_chunk(st, row, chunk, a);
      const float4 b = *reinterpret_cast<const float4*>(W + (size_t)(n0 + row) * ldw + k0 + 4 * chunk);
      ctd_tc_stage_chunk(st + CTD_TC_TERMS * CTD_TC_TILE_BYTES, row, chunk, b);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the tensor core
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a0 = ctd_smem_u32(st), b0 = a0 + CTD_TC_TERMS * CTD_TC_TILE_BYTES;
#pragma unroll
      for (int kk = 0; kk < CTD_TC_BK / 8; ++kk) {  // K = 8 per instruction = two 16-byte core columns
        const uint32_t ko = (uint32_t)kk * 256;
        const uint32_t tmem_acc = tmem_d + (uint32_t)((kk % CTD_TC_ACCS) * 128);   // K slice kk of every stage -> accumulator kk
        uint32_t acc = (uint32_t)(s != 0 || kk >= CTD_TC_ACCS);
        // smallest products first: (i, j) with i + j = 2, then 1, then 0
#pragma unroll
        for (int sum = CTD_TC_TERMS - 1; sum >= 0; --sum)
#pragma unroll
          for (int i = 0; i <= sum; ++i) {
            const int j = sum - i;
            ctd_umma_tf32(tmem_acc, ctd_umma_desc(a0 + i * CTD_TC_TILE_BYTES + ko, 128, 1024),
                          ctd_umma_desc(b0 + j * CTD_TC_TILE_BYTES + ko, 128, 1024), acc);
            acc = 1;
          }
      }
      // arrives on the stage barrier when every MMA issued so far has completed (implies fence::before_thread_sync)
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(ctd_smem_u32(&bars[buf])) : "memory");
    }
  }
  // the last commit covers all earlier MMAs
  {
    const int last = stages - 1;
    ok = ctd_mbar_wait(&bars[last & 1], (uint32_t)((last >> 1) & 1), err) && ok;
  }
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // ---- epilogue: TMEM -> registers -> bias / ReLU -> global; warp w owns lanes 32w..32w+31, one row per thread
  const int row = m0 + tid;
#pragma unroll 1
  for (int c0 = 0; c0 < CTD_TC_BN; c0 += 32) {
    uint32_t v[32];
    float sum[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) sum[j] = 0.f;
#pragma unroll 1
    for (int ai = 0; ai < CTD_TC_ACCS; ++ai) {
    const uint32_t taddr = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(ai * 128 + c0);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) sum[j] += __uint_as_float(v[j]);
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(sum[j]);
    if (ok && row < M) {
      float* y = Y + (size_t)row * ldy + n0 + c0;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        float4 o;
        o.x = __uint_as_float(v[j + 0]) + bias[n0 + c0 + j + 0];
        o.y = __uint_as_float(v[j + 1]) + bias[n0 + c0 + j + 1];
        o.z = __uint_as_float(v[j + 2]) + bias[n0 + c0 + j + 2];
        o.w = __uint_as_float(v[j + 3]) + bias[n0 + c0 + j + 3];
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        *reinterpret_cast<float4*>(y + j) = o;
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)(128 * CTD_TC_ACCS)));
}

// ---- the same product with the WEIGHT operand brought in by the TMA engine -------------------------------------------------
// The weights are static: ctd_set_value_model splits them into their three TF32 terms ONCE (ctd_k_split3, the same cvt.rna the
// kernel above applies to every operand on every launch) and keeps them as a [3][N][K] fp32 tensor with a 3-D tensor map
// (K, N, term).  A stage's B operand is then 24 bulk tensor copies of 128 rows x 16 bytes (one per term and 16-byte K chunk:
// cp.async.bulk.tensor.3d, SASS UTMALDG) issued by one thread and landing on the stage's `full` mbarrier (expect_tx = 48 KB),
// while all four warps stage the activation operand as before.  A box of 128 rows x 16 bytes lands as sixteen stacked 8-row core
// matrices, so the B descriptors use SBO = 128 B (8-row groups) and LBO = 2048 B (K-adjacent chunks); A keeps 1024 / 128.
__global__ void ctd_k_split3(const float* __restrict__ w, float* __restrict__ out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float a, b, c;
  ctd_tc_split3(w[i], a, b, c);
  out[i] = a; out[n + i] = b; out[2 * n + i] = c;
}
__device__ __forceinline__ void ctd_tma_load_3d(uint32_t smem_dst, const CUtensorMap* map, uint32_t mbar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_dst), "l"((uint64_t)map), "r"(mbar), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__global__ void __launch_bounds__(128) ctd_k_linear_tc_tma(const float* __restrict__ X, int ldx, const __grid_constant__ CUtensorMap wmap,
                                                           const float* __restrict__ bias, float* __restrict__ Y, int ldy, int M, int K,
                                                           int relu, int* err) {
  extern __shared__ uint8_t tc_smem_raw[];
  __shared__ uint64_t bars[2];    // stage free again: the MMAs that read it have completed (tcgen05.commit)
  __shared__ uint64_t full[2];    // stage's weight tiles have landed (TMA complete_tx)
  __shared__ uint32_t tmem_base_slot;
  uint8_t* smem = (uint8_t*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int m0 = blockIdx.x * CTD_TC_BM, n0 = blockIdx.y * CTD_TC_BN;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(ctd_smem_u32(&tmem_base_slot)), "r"((uint32_t)(128 * CTD_TC_ACCS)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    ctd_mbar_init(&bars[0], 1); ctd_mbar_init(&bars[1], 1);
    ctd_mbar_init(&full[0], 1); ctd_mbar_init(&full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = tmem_base_slot;
  const int stages = K / CTD_TC_BK;
  bool ok = true;
  for (int s = 0; s < stages; ++s) {
    const int buf = s & 1;
    uint8_t* st = smem + buf * CTD_TC_STAGE_BYTES;
    if (s >= 2) ok = ctd_mbar_wait(&bars[buf], (uint32_t)(((s >> 1) - 1) & 1), err) && ok;  // MMAs of slice s-2 are done
    const int k0 = s * CTD_TC_BK;
    if (tid == 0) {   // the weight operand: 3 terms x 8 chunks of 128 rows x 16 bytes
      const uint32_t fb = ctd_smem_u32(&full[buf]);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"((uint32_t)(CTD_TC_TERMS * CTD_TC_TILE_BYTES)) : "memory");
      const uint32_t b0 = ctd_smem_u32(st) + CTD_TC_TERMS * CTD_TC_TILE_BYTES;
#pragma unroll 1
      for (int t = 0; t < CTD_TC_TERMS; ++t)
#pragma unroll 1
        for (int c = 0; c < CTD_TC_BK / 4; ++c)
          ctd_tma_load_3d(b0 + t * CTD_TC_TILE_BYTES + c * 2048, &wmap, fb, k0 + 4 * c, n0, t);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {   // the activation operand: load, split, store in the UMMA layout
      const int idx = tid + 128 * i, row = idx >> 3, chunk = idx & 7;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + row < M) a = *reinterpret_cast<const float4*>(X + (size_t)(m0 + row) * ldx + k0 + 4 * chunk);
      ctd_tc_stage_chunk(st, row, chunk, a);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      ok = ctd_mbar_wait(&full[buf], (uint32_t)((s >> 1) & 1), err) && ok;   // the weight tiles are in
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a0 = ctd_smem_u32(st), b0 = a0 + CTD_TC_TERMS * CTD_TC_TILE_BYTES;
#pragma unroll
      for (int kk = 0; kk < CTD_TC_BK / 8; ++kk) {
        const uint32_t tmem_acc = tmem_d + (uint32_t)((kk % CTD_TC_ACCS) * 128);
        uint32_t acc = (uint32_t)(s != 0 || kk >= CTD_TC_ACCS);
#pragma unroll
        for (int sum = CTD_TC_TERMS - 1; sum >= 0; --sum)
#pragma unroll
          for (int i = 0; i <= sum; ++i) {
            const int j = sum - i;
            ctd_umma_tf32(tmem_acc, ctd_umma_desc(a0 + i * CTD_TC_TILE_BYTES + (uint32_t)kk * 256, 128, 1024),
                          ctd_umma_desc(b0 + j * CTD_TC_TILE_BYTES + (uint32_t)kk * 4096, 2048, 128), acc);
            acc = 1;
          }
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(ctd_smem_u32(&bars[buf])) : "memory");
    }
  }
  {
    const int last = stages - 1;
    ok = ctd_mbar_wait(&bars[last & 1], (uint32_t)((last >> 1) & 1), err) && ok;
  }
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int row = m0 + tid;
#pragma unroll 1
  for (int c0 = 0; c0 < CTD_TC_BN; c0 += 32) {
    uint32_t v[32];
    float sum[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) sum[j] = 0.f;
#pragma unroll 1
    for (int ai = 0; ai < CTD_TC_ACCS; ++ai) {
      const uint32_t taddr = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(ai * 128 + c0);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
            "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
            "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
            "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 32; ++j) sum[j] += __uint_as_float(v[j]);
    }
    if (ok && row < M) {
      float* y = Y + (size_t)row * ldy + n0 + c0;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        float4 o;
        o.x = sum[j + 0] + bias[n0 + c0 + j + 0];
        o.y = sum[j + 1] + bias[n0 + c0 + j + 1];
        o.z = sum[j + 2] + bias[n0 + c0 + j + 2];
        o.w = sum[j + 3] + bias[n0 + c0 + j + 3];
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        *reinterpret_cast<float4*>(y + j) = o;
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)(128 * CTD_TC_ACCS)));
}

// fc4 (128 -> 6) and model_reward_weights * square_and_normalize (train_utils.py:143-145): one row per thread
__global__ void __launch_bounds__(128) ctd_k_value_head(const float* __restrict__ H3, const float* __restrict__ w4t,
                                                        const float* __restrict__ b4, const uint8_t* __restrict__ pending,
                                                        uint32_t n, float* __restrict__ pred, float weight) {
  __shared__ float w[128 * 6 + 6];
  for (int i = threadIdx.x; i < 128 * 6; i += 128) w[i] = w4t[i];
  if (threadIdx.x < 6) w[768 + threadIdx.x] = b4[threadIdx.x];
  __syncthreads();
  const uint32_t r = blockIdx.x * 128 + threadIdx.x;
  if (r >= n || (pending != nullptr && !pending[r])) return;
  float y[6] = {w[768], w[769], w[770], w[771], w[772], w[773]};
  const float4* h4 = reinterpret_cast<const float4*>(H3 + (size_t)r * 128);
  for (int k4 = 0; k4 < 32; ++k4) {
    const float4 h = h4[k4];
    const float hv[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int o = 0; o < 6; ++o) y[o] = fmaf(w[(4 * k4 + j) * 6 + o], hv[j], y[o]);
  }
  float s = 0.f;
#pragma unroll
  for (int o = 0; o < 6; ++o) { y[o] *= y[o]; s += y[o]; }
#pragma unroll
  for (int o = 0; o < 6; ++o) pred[(size_t)r * 8 + o] = weight * (y[o] / s);
}
