// tcgen05 (5th-gen tensor core) 3xTF32 linear layer for the width-128 GraphNet MLPs.
//
//   Y[M,128] = epilogue( A[M,128] * B^T ),  B = W[128,128]  (or W^T for the data gradient)
//
// fp32 parity (1e-5 on logits/gradients) rules out a single TF32 pass (SURVEY.md 0.2), so
// every operand is split a = hi + lo with hi = tf32(a), lo = tf32(a - hi) and each product
// is three kind::tf32 MMAs (lo*hi, hi*lo, hi*hi) accumulated in fp32 in TMEM (measured
// error ~9e-7 rel-L2 per GEMM vs 2e-7 for fp32 FMA; end-to-end gradients stay under 1e-5).
//
// One persistent CTA per SM, 16 warps in 4 warpgroups, three roles connected by mbarriers
// (register budget rebalanced with setmaxnreg: loaders 64, MMA group 40, epilogue 192):
//   warps 0-3   loaders  : warp q owns rows 32q..32q+31 of every tile (= its TMEM lane quarter).
//                          K-blocks (32 rows x 128 B) are copied global -> smem with cp.async
//                          (no registers, no scoreboard coupling) into a ring of 3 private
//                          transpose tiles, so 48 KB per SM is always in flight; the warp then
//                          reads its tile with thread = row, splits hi/lo and writes the A operand
//                          straight into TMEM with tcgen05.st (4 stages x {hi,lo} x 32 columns).
//   warp  4     MMA      : one thread issues tcgen05.mma (M=128,N=128,K=8) with A from TMEM and B
//                          from smem descriptors; B (the weights, hi+lo = 128 KB, K-major
//                          SWIZZLE_128B) is built once per CTA and stays resident, so the only
//                          shared-memory traffic of the MMAs is the weight reads.  Accumulators are
//                          double-buffered in TMEM (2 x 128 columns).
//   warps 8-15  epilogue : two groups, group e drains accumulator buffer e (alternate tiles), so a
//                          tile's epilogue may take two MMA periods.  tcgen05.ld (thread = row),
//                          row-domain math (bias, LayerNorm statistics, dot), warp-local transpose
//                          through smem, then coalesced 128-bit global traffic for addends /
//                          residual / output; the global loads of a chunk are issued as one batch,
//                          one chunk ahead.
//
// Reference semantics covered (models/MLP.py:24-37, models/GNN.py:57-64, 95-104, 289-295):
//   MODE_ELEMENTWISE: y = act(acc + bias + addend[m] + g0[i0[m]] + g1[i1[m]]) + residual[m],  or  y *= (mask[m] > 0)
//   MODE_LAYERNORM  : y = LayerNorm(acc + bias) * gamma + beta + residual[m]
//   MODE_RELU_DOT   : y[m] = relu(acc + bias) . w + b          (decoder tail, out_channels = 1)
#include "common.cuh"

namespace gnc {
namespace tc {

constexpr int kTileM = 128;
constexpr int kD = 128;
constexpr int kKB = 32;                 // fp32 elements per K-block = one 128-byte swizzle row
constexpr int kNumKB = kD / kKB;        // 4
constexpr int kAStages = 4;             // TMEM A-operand stages
constexpr int kBlockBytes = kTileM * kKB * 4;   // 16 KB: one weight K-block image
constexpr int kLoaderWarps = 4;                     // warps 0..3: one per TMEM lane quarter
constexpr int kLoadBufs = 3;                        // cp.async transpose tiles in flight per loader warp
constexpr int kMmaWarp = kLoaderWarps;              // warp 4 (warps 5-7 pad the warpgroup)
constexpr int kEpiWarp0 = kLoaderWarps + 4;         // warps 8..15
constexpr int kEpiGroups = 2;
constexpr int kEpiWarps = 4 * kEpiGroups;
constexpr int kThreads = (kLoaderWarps + 4 + kEpiWarps) * 32;   // 512
constexpr int kRegsLaunch = 128;        // 65536 / 512 threads
constexpr int kRegsLoader = 64, kRegsMma = 40, kRegsEpi = 192;
// setmaxnreg moves registers inside the pool the CTA was LAUNCHED with (threads x launch
// registers), not the whole SM file: an inc that does not fit blocks forever.
static_assert(32 * (kLoaderWarps * kRegsLoader + 4 * kRegsMma + kEpiWarps * kRegsEpi) <= kThreads * kRegsLaunch,
              "setmaxnreg budget exceeds the CTA's register pool");
constexpr int kStagePitch = 36;         // floats per staged row (16-byte aligned, conflict-free)
constexpr int kTmemCols = 512;          // [0,256): two fp32 accumulators; [256,512): 4 A stages x (hi 32 | lo 32)
constexpr int kTmemA = 256;

// shared memory map (bytes, from a 1024-aligned base)
constexpr int kOffWhi = 0;
constexpr int kOffWlo = kOffWhi + kNumKB * kBlockBytes;                   //  65536
constexpr int kOffXpose = kOffWlo + kNumKB * kBlockBytes;                 // 131072: loader transpose tiles
constexpr int kOffStage = kOffXpose + kLoaderWarps * kLoadBufs * 32 * kStagePitch * 4; // 186368: epilogue transpose tiles
constexpr int kOffConst = kOffStage + kEpiWarps * 32 * kStagePitch * 4;   // 223232: bias,gamma,beta,dotw
constexpr int kOffBar = kOffConst + 4 * kD * 4;                           // 225280
constexpr int kSmemBytes = kOffBar + 128 + 1024;                          // + alignment slack = 226432

enum { MODE_ELEMENTWISE = 0, MODE_LAYERNORM = 1, MODE_RELU_DOT = 2 };

struct Params {
  const float* A; long long lda; long long M;
  const float* W; long long ldw; int transpose_w;
  const float* bias;
  const float* addend; long long ld_addend;
  const float* g0; const int32_t* i0; long long ld_g0;
  const float* g1; const int32_t* i1; long long ld_g1;
  int relu;
  const float* gamma; const float* beta; float eps;
  const float* residual; long long ld_res; const int32_t* res_idx;
  const float* mask; long long ld_mask;
  const float* dot_w; const float* dot_b;
  float* Y; long long ldy;
  float* ln_z; long long ld_ln_z; float* ln_mean; float* ln_rstd;   // LayerNorm epilogue: what its backward needs
  long long num_tiles;
  // co-scheduled weight sets (plain epilogue): CTA b uses set b % nsets and walks the tiles of
  // group b / nsets, so the nsets CTAs of a group read the same A tiles at the same time (L2 reuse)
  int nsets;
  const float* W_alt[2]; long long ldw_alt[2]; float* Y_alt[2];
};

// ---- PTX wrappers ---------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x989680;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand from tensor memory (lane = row, one 32-bit column per K element), B from smem
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* r) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(r);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
      "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* r) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
        "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
        "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"):
// rows of 128 bytes, 8-row groups 1024 bytes apart (SBO), swizzle applied by the hardware.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);         // start address
  d |= (uint64_t)1 << 16;                          // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                          // descriptor version
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
  return d;
}
// kind::tf32, fp32 accumulate, A and B K-major, M = 128, N = 128
constexpr uint32_t kInstrDesc = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// byte offset of (row, 16-byte chunk) inside one 16 KB K-block image
__device__ __forceinline__ uint32_t swz_off(int row, int chunk) {
  return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((chunk ^ (row & 7)) << 4));
}

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
__device__ __forceinline__ void split4(const float4& v, float4& hi, float4& lo) {
  hi.x = tf32_rna(v.x); hi.y = tf32_rna(v.y); hi.z = tf32_rna(v.z); hi.w = tf32_rna(v.w);
  lo.x = tf32_rna(v.x - hi.x); lo.y = tf32_rna(v.y - hi.y); lo.z = tf32_rna(v.z - hi.z); lo.w = tf32_rna(v.w - hi.w);
}
__device__ __forceinline__ void sts128(uint32_t saddr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- the kernel -------------------------------------------------------------------
template <int REGS>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS)); }
template <int REGS>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS)); }

__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) tc_linear_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wsel = p.nsets > 1 ? (int)(blockIdx.x % p.nsets) : 0;
  const float* Wsel = wsel == 0 ? p.W : p.W_alt[wsel - 1];
  const long long ldw_sel = wsel == 0 ? p.ldw : p.ldw_alt[wsel - 1];
  float* Ysel = wsel == 0 ? p.Y : p.Y_alt[wsel - 1];
  float* s_const = reinterpret_cast<float*>(sm + kOffConst);
  const uint32_t bar0 = base + kOffBar;
  // barrier slots (8 bytes each): a_full[4] a_empty[4] d_full[2] d_empty[2]; then the TMEM base pointer
  auto a_full = [&](int s) { return bar0 + 8u * s; };
  auto a_empty = [&](int s) { return bar0 + 32u + 8u * s; };
  auto d_full = [&](int d) { return bar0 + 64u + 8u * d; };
  auto d_empty = [&](int d) { return bar0 + 80u + 8u * d; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar + 96);

  // ---- one-time setup ----------------------------------------------------------
  if (threadIdx.x == 0) {
    for (int s = 0; s < kAStages; ++s) { mbar_init(a_full(s), kLoaderWarps * 32); mbar_init(a_empty(s), 1); }
    for (int d = 0; d < 2; ++d) { mbar_init(d_full(d), 1); mbar_init(d_empty(d), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {   // the MMA warp owns the TMEM allocation (all 512 columns: one CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // resident B operand: hi/lo images of W (row n = output feature, K-major), or of W^T
  for (int item = threadIdx.x; item < kD * kNumKB * 8; item += kThreads) {
    const int c = item & 7, n = (item >> 3) & (kD - 1), kb = item >> 10;
    const int k0 = kb * kKB + c * 4;
    float4 v;
    if (!p.transpose_w) {
      v = __ldg(reinterpret_cast<const float4*>(Wsel + (long long)n * ldw_sel + k0));
    } else {
      v.x = __ldg(Wsel + (long long)(k0 + 0) * ldw_sel + n);
      v.y = __ldg(Wsel + (long long)(k0 + 1) * ldw_sel + n);
      v.z = __ldg(Wsel + (long long)(k0 + 2) * ldw_sel + n);
      v.w = __ldg(Wsel + (long long)(k0 + 3) * ldw_sel + n);
    }
    float4 hi, lo;
    split4(v, hi, lo);
    const uint32_t off = (uint32_t)kb * kBlockBytes + swz_off(n, c);
    sts128(base + kOffWhi + off, hi);
    sts128(base + kOffWlo + off, lo);
  }
  for (int i = threadIdx.x; i < kD; i += kThreads) {
    s_const[i] = p.bias ? __ldg(p.bias + i) : 0.f;
    s_const[kD + i] = p.gamma ? __ldg(p.gamma + i) : 1.f;
    s_const[2 * kD + i] = p.beta ? __ldg(p.beta + i) : 0.f;
    s_const[3 * kD + i] = p.dot_w ? __ldg(p.dot_w + i) : 0.f;
  }
  fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long first = p.nsets > 1 ? blockIdx.x / p.nsets : blockIdx.x;
  const long long step = p.nsets > 1 ? gridDim.x / p.nsets : gridDim.x;
  const long long n_my = (p.num_tiles > first) ? (p.num_tiles - first + step - 1) / step : 0;

  if (warp < kLoaderWarps) {
    // ======================= loaders =======================
    reg_dec<kRegsLoader>();
    const int q = warp;                             // TMEM lane quarter = 32-row slice of the tile
    float* xp0 = reinterpret_cast<float*>(sm + kOffXpose) + warp * kLoadBufs * 32 * kStagePitch;
    const int rl = lane >> 3, c = lane & 7;
    const long long total = n_my * kNumKB;
    // copy K-block `it` (32 rows x 128 B) into transpose tile `b`; rows past M are zero-filled
    auto issue = [&](long long it, int b) {
      if (it < total) {
        const long long tile = first + (it >> 2) * step;
        const int kb = (int)(it & 3);
        const long long row0 = tile * kTileM + q * 32;
        const uint32_t dst0 = smem_u32(xp0 + b * 32 * kStagePitch) + (uint32_t)(rl * kStagePitch + c * 4) * 4u;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long row = row0 + i * 4 + rl;
          const long long rc = row < p.M ? row : p.M - 1;
          const uint32_t nbytes = row < p.M ? 16u : 0u;
          const float* src = p.A + rc * p.lda + kb * kKB + c * 4;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)(i * 4 * kStagePitch * 4)),
                       "l"(src), "r"(nbytes) : "memory");
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");     // always commit: uniform group counting
    };
#pragma unroll
    for (int b = 0; b < kLoadBufs; ++b) issue(b, b);
    int b = 0;
    for (long long it = 0; it < total; ++it) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kLoadBufs - 1) : "memory");   // K-block `it` has landed
      __syncwarp();
      const float* xp = xp0 + b * 32 * kStagePitch;
      const int s = (int)(it & 3);
      const uint32_t ph = (uint32_t)((it >> 2) & 1);
      mbar_wait(a_empty(s), ph ^ 1u);               // in-order single producer: at most one phase ahead
      tc_fence_after();
      const uint32_t ta = tmem_base + kTmemA + (uint32_t)s * 64 + ((uint32_t)(q * 32) << 16);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 x = *reinterpret_cast<const float4*>(xp + lane * kStagePitch + half * 16 + 4 * j);
          float4 h4, l4;
          split4(x, h4, l4);
          hi[4 * j] = h4.x; hi[4 * j + 1] = h4.y; hi[4 * j + 2] = h4.z; hi[4 * j + 3] = h4.w;
          lo[4 * j] = l4.x; lo[4 * j + 1] = l4.y; lo[4 * j + 2] = l4.z; lo[4 * j + 3] = l4.w;
        }
        tmem_st16(ta + half * 16, hi);
        tmem_st16(ta + 32 + half * 16, lo);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(a_full(s));
      __syncwarp();                                 // every lane has read the tile: refill it
      issue(it + kLoadBufs, b);
      b = (b + 1 == kLoadBufs) ? 0 : b + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp < kEpiWarp0) {
    // ======================= MMA issuer (warp 4; warps 5-7 pad the warpgroup) =======================
    reg_dec<kRegsMma>();
    if (warp == kMmaWarp && lane == 0) {
      // descriptors differ only in the 14-bit start-address field: derive them from one base
      // (keeps the issuing thread's live state tiny - it runs with a 40-register budget)
      const uint64_t desc_b0 = make_desc(base + kOffWhi);
      constexpr uint64_t kLoDelta = (uint64_t)((kOffWlo - kOffWhi) >> 4);
      long long it = 0, tcount = 0;
#pragma unroll 1
      for (long long tile = first; tile < p.num_tiles; tile += step, ++tcount) {
        const int d = (int)(tcount & 1);
        const uint32_t dph = (uint32_t)((tcount >> 1) & 1);
        mbar_wait(d_empty(d), dph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)d * kD;
#pragma unroll 1
        for (int kb = 0; kb < kNumKB; ++kb, ++it) {
          const int s = (int)(it & 3);
          const uint32_t ph = (uint32_t)((it >> 2) & 1);
          mbar_wait(a_full(s), ph);
          tc_fence_after();
          const uint32_t a_hi = tmem_base + kTmemA + (uint32_t)s * 64;
          const uint32_t a_lo = a_hi + 32;
          const uint64_t dkb = desc_b0 + (uint64_t)((kb * kBlockBytes) >> 4);
#pragma unroll
          for (int k = 0; k < kKB / 8; ++k) {
            const uint64_t dbh = dkb + (uint64_t)(k * 2);   // 8 tf32 = 32 bytes along K inside the swizzle row
            const uint64_t dbl = dbh + kLoDelta;
            // smallest terms first.  (A 4th lo*lo pass was measured: no accuracy gain - the
            // residual ~9e-7 rel-L2 is the tensor core's accumulation rounding, not the split.)
            umma_tf32_ts(d_tmem, a_lo + 8 * k, dbh, kInstrDesc, (kb | k) != 0);
            umma_tf32_ts(d_tmem, a_hi + 8 * k, dbl, kInstrDesc, 1);
            umma_tf32_ts(d_tmem, a_hi + 8 * k, dbh, kInstrDesc, 1);
          }
          umma_commit(a_empty(s));      // TMEM A stage reusable once these MMAs have read it
        }
        umma_commit(d_full(d));         // accumulator complete
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    reg_inc<kRegsEpi>();
    const int eg = (warp - kEpiWarp0) >> 2;         // epilogue group = accumulator buffer it drains
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    float* stg = reinterpret_cast<float*>(sm + kOffStage) + (warp - kEpiWarp0) * 32 * kStagePitch;
    const float* s_bias = s_const;
    const float* s_gamma = s_const + kD;
    const float* s_beta = s_const + 2 * kD;
    const float* s_dotw = s_const + 3 * kD;
    const int c4 = lane & 7, rl = lane >> 3;        // coalesced domain: 8 lanes per row, 4 rows per pass
    const uint32_t taddr = tmem_base + (uint32_t)eg * kD + ((uint32_t)(q * 32) << 16);
    long long k_tile = 0;                           // tiles drained by this group so far
    for (long long tcount = eg; tcount < n_my; tcount += kEpiGroups, ++k_tile) {
      const long long tile = first + tcount * step;
      const uint32_t dph = (uint32_t)(k_tile & 1);
      const long long wrow0 = tile * kTileM + q * 32;     // first global row of this warp
      // rows this lane touches in the coalesced domain (clamped: loads stay in bounds, stores are guarded)
      long long grow[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const long long g = wrow0 + j * 4 + rl;
        grow[j] = g < p.M ? g : p.M - 1;
      }

      if constexpr (MODE == MODE_ELEMENTWISE) {
        int gi0[8], gi1[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          gi0[j] = p.g0 ? __ldg(p.i0 + grow[j]) : 0;
          gi1[j] = p.g1 ? __ldg(p.i1 + grow[j]) : 0;
        }
        const bool has_ext = p.addend || p.g0 || p.g1;
        // ext[j] = sum of the pre-activation addends of (row j, this lane's 4 columns) for one chunk
        auto load_ext = [&](int ch, float4* ext) {
          const int col = ch * 32 + c4 * 4;
          if (p.g0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) ext[j] = __ldg(reinterpret_cast<const float4*>(p.g0 + (long long)gi0[j] * p.ld_g0 + col));
          } else if (p.addend) {
#pragma unroll
            for (int j = 0; j < 8; ++j) ext[j] = ldg_stream(reinterpret_cast<const float4*>(p.addend + grow[j] * p.ld_addend + col));
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) ext[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          if (p.g1) {
            float4 t[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) t[j] = __ldg(reinterpret_cast<const float4*>(p.g1 + (long long)gi1[j] * p.ld_g1 + col));
#pragma unroll
            for (int j = 0; j < 8; ++j) add4(ext[j], t[j]);
          }
          if (p.g0 && p.addend) {
            float4 t[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) t[j] = ldg_stream(reinterpret_cast<const float4*>(p.addend + grow[j] * p.ld_addend + col));
#pragma unroll
            for (int j = 0; j < 8; ++j) add4(ext[j], t[j]);
          }
        };
        float4 ext[8];
        if (has_ext) load_ext(0, ext);                 // overlaps the wait for the accumulator
        mbar_wait(d_full(eg), dph);
        tc_fence_after();
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
          {
            float r[32];
            tmem_ld32(taddr + ch * 32, r);
            tmem_ld_wait();
            if (ch == 3) { tc_fence_before(); mbar_arrive(d_empty(eg)); }   // accumulator drained
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(stg + lane * kStagePitch + 4 * j) = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
          }
          __syncwarp();
          const int col = ch * 32 + c4 * 4;
          const float4 b4 = *reinterpret_cast<const float4*>(s_bias + col);
          float4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            v[j] = *reinterpret_cast<const float4*>(stg + (j * 4 + rl) * kStagePitch + 4 * c4);
            add4(v[j], b4);
            if (has_ext) add4(v[j], ext[j]);
          }
          __syncwarp();                                // staging tile free for the next chunk
          if (p.residual) {
#pragma unroll
            for (int j = 0; j < 8; ++j) ext[j] = ldg_stream(reinterpret_cast<const float4*>(p.residual + grow[j] * p.ld_res + col));
          } else if (p.mask) {
#pragma unroll
            for (int j = 0; j < 8; ++j) ext[j] = ldg_stream(reinterpret_cast<const float4*>(p.mask + grow[j] * p.ld_mask + col));
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (p.relu) { v[j].x = fmaxf(v[j].x, 0.f); v[j].y = fmaxf(v[j].y, 0.f); v[j].z = fmaxf(v[j].z, 0.f); v[j].w = fmaxf(v[j].w, 0.f); }
            if (p.residual) add4(v[j], ext[j]);
            else if (p.mask) {      // ReLU backward of the layer that produced this operand: y *= (mask > 0)
              v[j].x = ext[j].x > 0.f ? v[j].x : 0.f; v[j].y = ext[j].y > 0.f ? v[j].y : 0.f;
              v[j].z = ext[j].z > 0.f ? v[j].z : 0.f; v[j].w = ext[j].w > 0.f ? v[j].w : 0.f;
            }
            if (wrow0 + j * 4 + rl < p.M) stg_stream(reinterpret_cast<float4*>(Ysel + grow[j] * p.ldy + col), v[j]);
          }
          if (has_ext && ch < 3) load_ext(ch + 1, ext); // next chunk's addends fly during the next TMEM read
        }
      } else if constexpr (MODE == MODE_RELU_DOT) {
        mbar_wait(d_full(eg), dph);
        tc_fence_after();
        float acc = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
          float r[32];
          tmem_ld32(taddr + ch * 32, r);
          tmem_ld_wait();
          if (ch == 3) { tc_fence_before(); mbar_arrive(d_empty(eg)); }
#pragma unroll
          for (int cidx = 0; cidx < 32; ++cidx)
            acc = fmaf(fmaxf(r[cidx] + s_bias[ch * 32 + cidx], 0.f), s_dotw[ch * 32 + cidx], acc);
        }
        const long long g = wrow0 + lane;
        if (g < p.M) Ysel[g * p.ldy] = acc + (p.dot_b ? __ldg(p.dot_b) : 0.f);
      } else {
        // LayerNorm.  Pass 1 over the accumulator: each 32-column chunk's mean and sum of squared
        // deviations from it (two sweeps over the chunk's registers), merged into the row's running
        // mean / M2 with Chan's pairwise update.  Every term is a deviation from a mean, so the
        // statistics are exact to fp32 rounding whatever the row's centre (a one-pass
        // E[z^2] - E[z]^2, even shifted by the first element, loses ~7 bits when that element
        // is an outlier of the row).  Pass 2 re-reads TMEM, normalises and stores.  No 128-register
        // row buffer.
        float4 res[8];
        long long rrow[8];                              // residual rows: identity, or a table lookup
#pragma unroll
        for (int j = 0; j < 8; ++j) rrow[j] = (p.residual && p.res_idx) ? (long long)__ldg(p.res_idx + grow[j]) : grow[j];
        if (p.residual) {                               // chunk 0 of the residual, ahead of the accumulator
#pragma unroll
          for (int j = 0; j < 8; ++j)
            res[j] = __ldg(reinterpret_cast<const float4*>(p.residual + rrow[j] * p.ld_res + c4 * 4));
        }
        mbar_wait(d_full(eg), dph);
        tc_fence_after();
        float mu = 0.f, m2 = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
          float r[32];
          tmem_ld32(taddr + ch * 32, r);
          tmem_ld_wait();
          float s = 0.f;
#pragma unroll
          for (int cidx = 0; cidx < 32; ++cidx) {
            r[cidx] += s_bias[ch * 32 + cidx];
            s += r[cidx];
          }
          const float mc = s * (1.0f / 32);
          float q = 0.f;
#pragma unroll
          for (int cidx = 0; cidx < 32; ++cidx) {
            const float dlt = r[cidx] - mc;
            q = fmaf(dlt, dlt, q);
          }
          // merge (32 ch columns, mean mu, M2 m2) with (32 columns, mean mc, M2 q)
          const float delta = mc - mu;
          const float inv_n = ch == 0 ? 1.0f : ch == 1 ? 0.5f : ch == 2 ? 1.0f / 3 : 0.25f;     // 1 / (ch + 1)
          const float w = ch == 0 ? 0.0f : ch == 1 ? 16.0f : ch == 2 ? 64.0f / 3 : 24.0f;    // 32 ch / (ch + 1)
          mu = fmaf(delta, inv_n, mu);
          m2 += fmaf(delta * delta, w, q);
        }
        const float var = m2 * (1.0f / kD);
        const float rs = 1.0f / sqrtf(var + p.eps);
        if (p.ln_mean && wrow0 + lane < p.M) {          // thread = row: the statistics the backward reuses
          p.ln_mean[wrow0 + lane] = mu;
          p.ln_rstd[wrow0 + lane] = rs;
        }
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
          {
            float r[32];
            tmem_ld32(taddr + ch * 32, r);
            tmem_ld_wait();
            if (ch == 3) { tc_fence_before(); mbar_arrive(d_empty(eg)); }
            if (p.ln_z) {
              // training: the pre-LayerNorm activation goes out too (same transpose through the staging tile), so
              // that no separate LayerNorm pass has to re-read it
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int cb = ch * 32 + 4 * j;
                *reinterpret_cast<float4*>(stg + lane * kStagePitch + 4 * j) =
                    make_float4(r[4 * j] + s_bias[cb], r[4 * j + 1] + s_bias[cb + 1], r[4 * j + 2] + s_bias[cb + 2], r[4 * j + 3] + s_bias[cb + 3]);
              }
              __syncwarp();
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 zz = *reinterpret_cast<const float4*>(stg + (j * 4 + rl) * kStagePitch + 4 * c4);
                if (wrow0 + j * 4 + rl < p.M) stg_stream(reinterpret_cast<float4*>(p.ln_z + grow[j] * p.ld_ln_z + ch * 32 + c4 * 4), zz);
              }
              __syncwarp();
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int cb = ch * 32 + 4 * j;
              float4 o;
              o.x = ((r[4 * j + 0] + s_bias[cb + 0]) - mu) * rs * s_gamma[cb + 0] + s_beta[cb + 0];
              o.y = ((r[4 * j + 1] + s_bias[cb + 1]) - mu) * rs * s_gamma[cb + 1] + s_beta[cb + 1];
              o.z = ((r[4 * j + 2] + s_bias[cb + 2]) - mu) * rs * s_gamma[cb + 2] + s_beta[cb + 2];
              o.w = ((r[4 * j + 3] + s_bias[cb + 3]) - mu) * rs * s_gamma[cb + 3] + s_beta[cb + 3];
              *reinterpret_cast<float4*>(stg + lane * kStagePitch + 4 * j) = o;
            }
          }
          __syncwarp();
          const int col = ch * 32 + c4 * 4;
          float4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            v[j] = *reinterpret_cast<const float4*>(stg + (j * 4 + rl) * kStagePitch + 4 * c4);
            if (p.residual) add4(v[j], res[j]);
          }
          __syncwarp();
          if (p.residual && ch < 3) {                   // next chunk's residual flies during these stores
#pragma unroll
            for (int j = 0; j < 8; ++j)
              res[j] = __ldg(reinterpret_cast<const float4*>(p.residual + rrow[j] * p.ld_res + col + 32));
          }
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (wrow0 + j * 4 + rl < p.M) stg_stream(reinterpret_cast<float4*>(Ysel + grow[j] * p.ldy + col), v[j]);
        }
      }
    }
  }

  // ---- teardown ---------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTmemCols) : "memory");
  }
}

template <int MODE>
static int launch(const Params& p, cudaStream_t st) {
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(tc_linear_kernel<MODE>, kSmemBytes, "tc_linear")) return rc_attr;
  long long grid = p.num_tiles < kNumSMs ? p.num_tiles : kNumSMs;
  if (p.nsets > 1) {
    long long groups = kNumSMs / p.nsets;
    if (groups > p.num_tiles) groups = p.num_tiles;
    grid = groups * p.nsets;
  }
  tc_linear_kernel<MODE><<<(unsigned)grid, kThreads, kSmemBytes, st>>>(p);
  return check_launch("tc_linear_kernel");
}

}  // namespace tc
}  // namespace gnc

using namespace gnc;

extern "C" int gnc_tc_linear_f32(const float* A, int64_t lda, int64_t M, int K, const float* W, int64_t ldw, int N,
                                 int transpose_w, const gnc_tc_epilogue_t* epi, float* Y, int64_t ldy,
                                 gnc_stream_t stream) {
  GNC_REQUIRE(K == tc::kD && N == tc::kD, "tc_linear: this engine is specialised for 128 x 128 weight tiles");
  GNC_REQUIRE(W && epi && M >= 0 && lda >= K && ldw >= tc::kD, "tc_linear: bad arguments");
  if (M == 0) return GNC_OK;                          // (empty tensors have no pointers: an edge-less graph)
  GNC_REQUIRE(A && Y, "tc_linear: null pointer");
  GNC_REQUIRE(lda % 4 == 0 && aligned16(A) && aligned16(W) && ldw % 4 == 0, "tc_linear: A / W rows must be 16-byte aligned");
  tc::Params p;
  p.A = A; p.lda = lda; p.M = M; p.W = W; p.ldw = ldw; p.transpose_w = transpose_w;
  p.bias = epi->bias;
  p.addend = epi->addend; p.ld_addend = epi->ld_addend;
  p.g0 = epi->gather0; p.i0 = epi->gather0_idx; p.ld_g0 = epi->ld_gather0;
  p.g1 = epi->gather1; p.i1 = epi->gather1_idx; p.ld_g1 = epi->ld_gather1;
  p.relu = epi->relu;
  p.gamma = epi->gamma; p.beta = epi->beta; p.eps = epi->eps;
  p.residual = epi->residual; p.ld_res = epi->ld_residual; p.res_idx = epi->residual_idx;
  p.mask = epi->mask; p.ld_mask = epi->ld_mask;
  p.dot_w = epi->dot_w; p.dot_b = epi->dot_b;
  p.Y = Y; p.ldy = ldy;
  p.ln_z = epi->ln_z; p.ld_ln_z = epi->ld_ln_z; p.ln_mean = epi->ln_mean; p.ln_rstd = epi->ln_rstd;
  p.nsets = 1;
  p.W_alt[0] = p.W_alt[1] = nullptr; p.ldw_alt[0] = p.ldw_alt[1] = 0; p.Y_alt[0] = p.Y_alt[1] = nullptr;
  p.num_tiles = (M + tc::kTileM - 1) / tc::kTileM;
  GNC_REQUIRE(!p.g0 || p.i0, "tc_linear: gather0 needs gather0_idx");
  GNC_REQUIRE(!p.g1 || p.i1, "tc_linear: gather1 needs gather1_idx");
  auto ok4 = [](const float* q, int64_t ld) { return !q || (aligned16(q) && ld % 4 == 0); };
  GNC_REQUIRE(!(p.mask && (p.residual || epi->gamma || epi->dot_w)), "tc_linear: mask combines with the elementwise epilogue only, without residual");
  GNC_REQUIRE(ok4(p.addend, p.ld_addend) && ok4(p.g0, p.ld_g0) && ok4(p.g1, p.ld_g1) && ok4(p.residual, p.ld_res) && ok4(p.mask, p.ld_mask),
              "tc_linear: addend / gather / residual rows must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (epi->dot_w) {
    GNC_REQUIRE(!epi->gamma && !p.addend && !p.g0 && !p.g1 && !p.residual && epi->relu && ldy >= 1,
                "tc_linear: dot epilogue = relu(acc + bias) . w only");
    return tc::launch<tc::MODE_RELU_DOT>(p, st);
  }
  GNC_REQUIRE(ldy >= tc::kD && ldy % 4 == 0 && aligned16(Y), "tc_linear: Y rows must be 16-byte aligned");
  GNC_REQUIRE(!epi->residual_idx || (epi->gamma && epi->residual), "tc_linear: residual_idx is supported by the LayerNorm epilogue only");
  if (epi->gamma) {
    GNC_REQUIRE(epi->beta && !p.addend && !p.g0 && !p.g1 && !epi->relu, "tc_linear: LayerNorm epilogue takes bias + residual only");
    GNC_REQUIRE(!p.ln_z || (aligned16(p.ln_z) && p.ld_ln_z >= tc::kD && p.ld_ln_z % 4 == 0), "tc_linear: ln_z rows must be 16-byte aligned");
    GNC_REQUIRE((p.ln_mean == nullptr) == (p.ln_rstd == nullptr), "tc_linear: ln_mean and ln_rstd come together");
    return tc::launch<tc::MODE_LAYERNORM>(p, st);
  }
  GNC_REQUIRE(!p.ln_z && !p.ln_mean && !p.ln_rstd, "tc_linear: ln_z / ln_mean / ln_rstd belong to the LayerNorm epilogue");
  return tc::launch<tc::MODE_ELEMENTWISE>(p, st);
}

// Y_s[M, 128] = A[M, 128] * W_s^T for 2 or 3 weight sets in ONE launch: the CTAs of a group walk
// the same row tiles at the same time, so A is fetched from HBM once and served to the other sets
// from L2 (the P / Q / T products of a GraphNet block all read the node latents).
extern "C" int gnc_tc_linear_multi_f32(const float* A, int64_t lda, int64_t M, int nsets, const float* const* W,
                                       const int64_t* ldw, float* const* Y, int64_t ldy, gnc_stream_t stream) {
  GNC_REQUIRE(nsets >= 2 && nsets <= 3 && A && W && ldw && Y && M >= 0 && lda >= tc::kD && ldy >= tc::kD,
              "tc_linear_multi: need 2 or 3 weight sets");
  if (M == 0) return GNC_OK;
  GNC_REQUIRE(lda % 4 == 0 && aligned16(A) && ldy % 4 == 0, "tc_linear_multi: rows must be 16-byte aligned");
  tc::Params p = {};
  p.A = A; p.lda = lda; p.M = M; p.transpose_w = 0;
  p.eps = 1e-5f; p.ldy = ldy;
  p.num_tiles = (M + tc::kTileM - 1) / tc::kTileM;
  p.nsets = nsets;
  for (int s = 0; s < nsets; ++s) {
    GNC_REQUIRE(W[s] && Y[s] && aligned16(W[s]) && aligned16(Y[s]) && ldw[s] % 4 == 0 && ldw[s] >= tc::kD,
                "tc_linear_multi: bad weight / output pointer");
    if (s == 0) { p.W = W[0]; p.ldw = ldw[0]; p.Y = Y[0]; }
    else { p.W_alt[s - 1] = W[s]; p.ldw_alt[s - 1] = ldw[s]; p.Y_alt[s - 1] = Y[s]; }
  }
  return tc::launch<tc::MODE_ELEMENTWISE>(p, (cudaStream_t)stream);
}
