// Chained width-128 MLP on tcgen05: two or three Linear(128,128) layers (+ ReLU between them, LayerNorm +
// residual or the decoder dot product at the end) evaluated in ONE kernel, the hidden activations
// never leaving the SM:
//
//   Y = tail( W2 relu( W1 relu( W0 A + b0 + G0[i0] + G1[i1] ) + b1 ) + b2 )
//
// This is the whole EdgeProcessor / NodeProcessor MLP of a GraphNet block (models/GNN.py:57-64, 95-104,
// models/MLP.py:24-37) in the restructured form of DESIGN.md section 4: the gathered addends are the
// per-node products P[row], Q[col] (edge model) or the plain addend T (node model).
//
// fp32 parity.  Operands are split into two fp16 pieces, a = a1 + a2 (22 significant bits), after an exact
// power-of-two scaling that keeps the second piece out of the fp16 subnormal range (weights x 2^8,
// activations x 2^4; the accumulator is scaled back by 2^-12 in the epilogue), and each product is three
// kind::f16 MMAs (a1 w2, a2 w1, a1 w1; the dropped a2 w2 is below 2^-22) accumulated in fp32 in TMEM.
// Measured 4.7e-7 rel-L2 per GEMM for |a| from 1e-2 to 2e2 (scripts/probes/pair_probe.cu) - tighter than
// 3xTF32 (9e-7) or bf16x3 with six products (8e-7) at HALF their tensor-pipe work and 2/3 of the bf16x3
// weight footprint.  Domain: |activation| < 4094 (fp16 overflow beyond it gives inf / NaN outputs).
//
// CTA pair.  Two CTAs of a cluster share every MMA (tcgen05.mma.cta_group::2, M = 256, N = 128): each CTA
// keeps the 64 output features n = 64 * rank .. 64 * rank + 63 of every layer in shared memory (32 KB per
// layer) and its own 128 rows of A and D in tensor memory, which leaves ~120 KB of shared memory per SM
// for the staging rings that hide the memory latency.  The leader CTA's single MMA thread issues for both.
//
// Per CTA: 16 warps.
//   warps 0-3   loaders  : cp.async 32 x 32 fp32 chunks of A (global -> swizzled smem), read back with
//                          thread = row, split, tcgen05.st into the A operand (2 pieces x 64 packed columns).
//   warp  4     MMA      : (leader) per layer and 32-wide K chunk: wait for the chunk, 6 MMAs.  Layer
//                          l+1's chunk c is produced by layer l's epilogue from accumulator columns
//                          32c..32c+31, so its MMAs overlap the rest of that epilogue.  Accumulators
//                          ping-pong between two 128-column TMEM buffers.
//   warps 8-15  epilogue : warp (q, h) owns rows 32q..32q+31 and columns 32c + 16h .. + 15 of every
//                          chunk.  Hidden layers: tcgen05.ld -> bias (+ addends staged through smem by
//                          the warp's own cp.async) -> ReLU -> split -> tcgen05.st as the next A.  Last
//                          layer: 64 values per thread in registers, exact two-pass LayerNorm statistics
//                          (halves combined through smem), residual, transpose through smem, coalesced
//                          stores.
#include <stdlib.h>

#include "common.cuh"

namespace gnc {
namespace chain {

constexpr int kD = 128;
constexpr int kTileM = 256;                       // rows per CTA-pair tile
constexpr int kMaxLayers = 3;
constexpr int kImgBytes = 64 * 128;               // one (piece, K-block) image: 64 weight rows x 64 fp16
constexpr int kLayerBytes = 4 * kImgBytes;        // 2 pieces x 2 K-blocks = 32 KB
constexpr int kLoaderWarps = 4, kLoadBufs = 3;
constexpr float kScaleW = 256.f, kScaleA = 16.f;  // exact power-of-two operand scalings
constexpr float kUnscaleD = 1.f / (kScaleW * kScaleA);
constexpr int kMmaWarp = 4;
constexpr int kEpiWarp0 = 8, kEpiWarps = 8;
constexpr int kThreads = 512;
constexpr int kRegsLoader = 72, kRegsMma = 40, kRegsEpi = 200;
static_assert(32 * (4 * kRegsLoader + 4 * kRegsMma + kEpiWarps * kRegsEpi) <= kThreads * 128, "setmaxnreg budget");

constexpr int kChunkBytes = 32 * 128;             // loader chunk: 32 rows x 32 fp32
constexpr int kSlotBytes = 32 * 64;               // epilogue tile: 32 rows x 16 fp32
constexpr int kOffW = 0;
constexpr int kEpiSlots = 4;                      // per epilogue warp: addends (P, Q) x 2 steps, or 4 residual steps
constexpr int kOffLd = kOffW + kMaxLayers * kLayerBytes;                    //  98304
constexpr int kOffEp = kOffLd + kLoaderWarps * kLoadBufs * kChunkBytes;      // 147456
constexpr int kOffConst = kOffEp + kEpiWarps * kEpiSlots * kSlotBytes;       // 212992: bias[3], gamma, beta
constexpr int kOffXchg = kOffConst + 5 * kD * 4;                             // 215552: 2 x [8 warps][32 lanes]
constexpr int kOffBar = kOffXchg + 2 * kEpiWarps * 32 * 4;                   // 217600
constexpr int kSmemBytes = kOffBar + 256 + 1024;                             // 218880

constexpr uint32_t kTmemD = 0;                    // two accumulators: [0,128) [128,256)
constexpr uint32_t kTmemA = 256;                  // A pieces: [256,320) [320,384); [384,512) is free

struct Params {
  const float* A; long long lda; long long M;
  int nlayers;
  const float* W[kMaxLayers]; long long ldw[kMaxLayers]; const float* bias[kMaxLayers];
  const float* g0; const int32_t* i0; long long ld_g0;
  const float* g1; const int32_t* i1; long long ld_g1;
  const float* gamma; const float* beta; float eps;
  const float* residual; const int32_t* res_idx; long long ld_res;
  const float* dot_w; const float* dot_b;
  float* Y; long long ldy;
  float* Ym[kMaxLayers];                      // multi mode: one output per weight set
  int multi;
  // pre-stage mode (A == NULL): the first operand is relu(g2[i2[m]] + g0[i0[m]] + g1[i1[m]] + pre_bias), built by
  // the epilogue warps - block 0 of the grid-graph path, whose edge latents are a 4-row table (models/GNN.py:57-64)
  const float* g2; const int32_t* i2; long long ld_g2; const float* pre_bias;
  // second operand of the first layer: z0 += A2 W_A2^T (the node processor's cat([x, agg]) without a T tensor)
  const float* A2; long long lda2; const float* W_A2; long long ldw_A2;
  // narrow first layer folded into the loader: the operand is relu(A[:, :syn_k] syn_W^T + syn_b), syn_k <= 8
  const float* syn_W; long long ld_syn_W; const float* syn_b; int syn_k;
  // aggregated first operand (two-operand node form): A is the EDGE-row table and row m of the first operand is the ordered
  // sum of A[agg_eid[k]], k in [agg_rowptr[m], agg_rowptr[m + 1]) - at most two entries per row (caller-checked)
  const int32_t* agg_rowptr; const int32_t* agg_eid;
  // paired destination slots (gnc_tc_chain_t): edge_slots 1 - a negative i0 marks a padding row (output +0.0), 2 - and Y
  // takes the pair sums (0 + y[2v]) + y[2v + 1]; paired (node form) - row m of the first operand is (0 + A[2m]) + A[2m + 1]
  int edge_slots; int paired;
  // training forward (two-tile kernel, Spec<1> / Spec<2>): a1, a2 (hidden ReLU outputs), z (LayerNorm input), row statistics
  float* st_a1; float* st_a2; float* st_z; long long ld_st; float* st_mean; float* st_rstd;
  long long num_tiles;
  unsigned long long* trace; int trace_cap;   // debug timeline of CTA 0 (gnc_debug_chain_trace), normally NULL
};
constexpr int kTraceRoles = 4;                // 0 MMA thread, 1 epilogue warp (q0,h0), 2 loader warp 0, 3 epilogue warp (q0,h1)

// ---- PTX wrappers ---------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// address of the same barrier in the leader CTA's shared memory (cluster window)
__device__ __forceinline__ uint32_t map_to_leader(uint32_t local) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(local));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  // default (.release.cta) semantics: the data handed over lives in tensor memory and is ordered by the
  // tcgen05 fences; the .release.cluster form costs a MEMBAR.ALL.GPU per arrive (measured: ~1400 cycles a chunk)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "CW_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x989680;\n\t"
      "@p bra.uni CW_DONE;\n\t"
      "bra.uni CW_LOOP;\n\t"
      "CW_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// A (fp16 pairs, K-major) from tensor memory, B from shared memory, both CTAs of the pair
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs once the MMAs issued so far retire
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* u) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(u[0]),
               "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* r) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory matrix descriptor (rows of 128 bytes, 8-row groups 1024 bytes apart)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16: fp16 x fp16 -> fp32, A and B K-major, M = 256 (the pair), N = 128.  (Issuing each layer as two
// N = 64 column halves, to overlap the first half's epilogue with the second half's MMAs, was measured:
// 12.6 ms instead of 9.2 ms on 16.6 M rows - the N = 64 shape runs well below the N = 128 rate.)
constexpr uint32_t kInstrDesc = (1u << 4) | (0u << 7) | (0u << 10) | ((128u >> 3) << 17) | ((256u >> 4) << 24);

// Packed FP32 (sm_100: FFMA2 / FADD2 / FMUL2 act on a 64-bit register pair).  Each lane is the scalar IEEE
// round-to-nearest operation without flush to zero, so two scalar operations and their packed form give the same
// bits as long as the order of operations is kept.  The per-element work of loaders and epilogues is written in
// pairs of adjacent columns with these; ReLU stays scalar (there is no packed max).
__device__ __forceinline__ float2 pair2(const float* v) { return make_float2(v[0], v[1]); }
__device__ __forceinline__ void set2(float* v, float2 r) { v[0] = r.x; v[1] = r.y; }
__device__ __forceinline__ float2 dup2(float s) { return make_float2(s, s); }

// (x0, x1), already scaled -> two packed fp16 pairs (low half = x0) with p1 + p2 == x to 22 bits.  The hi piece is
// unpacked with two cvt.f32.f16: there is no cheaper exact unpack; the residual x - h is one packed subtraction.
__device__ __forceinline__ void split2(float2 x, uint32_t& p1, uint32_t& p2) {
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(p1) : "f"(x.y), "f"(x.x));
  float h0, h1;
  asm("{.reg .f16 lo, hi; mov.b32 {lo, hi}, %2; cvt.f32.f16 %0, lo; cvt.f32.f16 %1, hi;}" : "=f"(h0), "=f"(h1) : "r"(p1));
  const float2 r = __fadd2_rn(x, make_float2(-h0, -h1));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(p2) : "f"(r.y), "f"(r.x));
}
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& p1, uint32_t& p2) { split2(make_float2(x0, x1), p1, p2); }
// (x0, x1) x s, s an exact power of two (the operand scalings), then split
__device__ __forceinline__ void split2_scaled(float x0, float x1, float s, uint32_t& p1, uint32_t& p2) {
  split2(__fmul2_rn(make_float2(x0, x1), dup2(s)), p1, p2);
}
// ReLU that keeps NaN (fmaxf would turn the NaN of an out-of-range fp16 operand into a silent 0)
__device__ __forceinline__ float relu_nan(float x) {
  float y;
  asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t nbytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
}
// L2 residency hints (two-tile kernel): the rows of A are read again ~2 tiles later as the residual; without a
// hint the P / Q gathers and the output stream push ~70 % of them out of L2 in between (ncu: DRAM reads 1.36 x
// algorithmic).  A rows are loaded evict_last, their second (last) read and the output stores are evict_first.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void cp_async16_hint(uint32_t dst, const void* src, uint32_t nbytes, uint64_t policy) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;" ::"r"(dst), "l"(src), "r"(nbytes), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void stg_hint(float4* p, const float4& v, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(policy)
               : "memory");
}
// 256-bit streaming load (sm_100: LDG.256): a lane reads 32 contiguous bytes of its own row
__device__ __forceinline__ void ldg256_stream(const float* p, float* v) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
// 256-bit store (sm_100: STG.256): a lane that owns 32 contiguous bytes of a row writes a whole sector per instruction
__device__ __forceinline__ void stg256(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }

template <int REGS>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS)); }
template <int REGS>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS)); }

// (clock << 8 | tag) records for one thread of a role; only CTA 0 traces.  Compiled out (ON = false) of
// the specialised instantiations.
template <bool ON>
struct Tracer {
  unsigned long long* buf; int cap; int n;
  __device__ __forceinline__ void init(const Params& p, int role, bool on) {
    if (ON) {
      buf = (on && p.trace && blockIdx.x == 0) ? p.trace + (size_t)role * p.trace_cap : nullptr;
      cap = p.trace_cap; n = 0;
    }
  }
  __device__ __forceinline__ void ev(int tag) {
    if (ON) {
      if (buf && n < cap) buf[n++] = ((unsigned long long)clock64() << 8) | (unsigned)tag;
    }
  }
};

// Compile-time view of a launch.  0 = absent, 1 = present, 2 = decided at run time.  The epilogue is
// bound by instruction issue, and the run-time-generic form spends ~45 % of its instructions on
// predication and re-derived addresses, so the shapes the GraphNet forward uses are specialised.
template <int SPEC> struct Spec { static constexpr int nl = 0, g0 = 2, i0 = 2, g1 = 2, i1 = 2, res = 2, ridx = 2, ln = 2, dot = 2; static constexpr bool trace = true, multi = false, pre = false; };
// edge processor: 3 layers, P[row] + Q[col], LayerNorm, residual          (models/GNN.py:57-64)
template <> struct Spec<1> { static constexpr int nl = 3, g0 = 1, i0 = 1, g1 = 1, i1 = 1, res = 1, ridx = 0, ln = 1, dot = 0; static constexpr bool trace = false, multi = false, pre = false; };
// node processor: 3 layers, one plain addend, LayerNorm, residual          (models/GNN.py:95-104)
template <> struct Spec<2> { static constexpr int nl = 3, g0 = 1, i0 = 0, g1 = 0, i1 = 0, res = 1, ridx = 0, ln = 1, dot = 0; static constexpr bool trace = false, multi = false, pre = false; };
// last two layers of a processor MLP: LayerNorm, residual (direct or through a table)
template <> struct Spec<3> { static constexpr int nl = 2, g0 = 0, i0 = 0, g1 = 0, i1 = 0, res = 1, ridx = 2, ln = 1, dot = 0; static constexpr bool trace = false, multi = false, pre = false; };
// last two layers of an encoder MLP: LayerNorm, no residual                  (models/GNN.py:262-287)
template <> struct Spec<4> { static constexpr int nl = 2, g0 = 0, i0 = 0, g1 = 0, i1 = 0, res = 0, ridx = 0, ln = 1, dot = 0; static constexpr bool trace = false, multi = false, pre = false; };
// decoder: two layers and the dot-product tail                               (models/GNN.py:289-295)
template <> struct Spec<5> { static constexpr int nl = 2, g0 = 0, i0 = 0, g1 = 0, i1 = 0, res = 0, ridx = 0, ln = 0, dot = 1; static constexpr bool trace = false, multi = false, pre = false; };
// multi mode: nl independent products of the SAME rows, Y_l = A W_l^T (the P / Q / T products of a block)
template <> struct Spec<6> { static constexpr int nl = 0, g0 = 0, i0 = 0, g1 = 0, i1 = 0, res = 0, ridx = 0, ln = 0, dot = 0; static constexpr bool trace = false, multi = true, pre = false; };
// pre-stage + two layers + LayerNorm + table residual: the block-0 edge processor of the grid-graph path
template <> struct Spec<7> { static constexpr int nl = 2, g0 = 1, i0 = 1, g1 = 1, i1 = 1, res = 1, ridx = 1, ln = 1, dot = 0; static constexpr bool trace = false, multi = false, pre = true; };
// Spec<1> with the timeline recorder compiled in (scripts/chain_trace.py)
template <> struct Spec<8> { static constexpr int nl = 3, g0 = 1, i0 = 1, g1 = 1, i1 = 1, res = 1, ridx = 0, ln = 1, dot = 0; static constexpr bool trace = true, multi = false, pre = false; };
#define GNC_FLAG(field, runtime) (Spec<SPEC>::field == 2 ? (runtime) : (Spec<SPEC>::field != 0))

// ---- the kernel -------------------------------------------------------------------
template <int SPEC>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) tc_chain_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nl = Spec<SPEC>::nl ? Spec<SPEC>::nl : p.nlayers;
  const bool has_g0 = GNC_FLAG(g0, p.g0 != nullptr), has_i0 = GNC_FLAG(i0, p.i0 != nullptr);
  const bool has_g1 = GNC_FLAG(g1, p.g1 != nullptr), has_i1 = GNC_FLAG(i1, p.i1 != nullptr);
  const bool has_res = GNC_FLAG(res, p.residual != nullptr), has_ridx = GNC_FLAG(ridx, p.res_idx != nullptr);
  const bool has_ln = GNC_FLAG(ln, p.gamma != nullptr), has_dot = GNC_FLAG(dot, p.dot_w != nullptr);
  using Trace = Tracer<Spec<SPEC>::trace>;
  constexpr bool kMulti = Spec<SPEC>::multi;
  constexpr bool kPre = Spec<SPEC>::pre;
  float* s_const = reinterpret_cast<float*>(sm + kOffConst);   // bias[0..2], gamma (or dot_w), beta
  const uint32_t bar0 = base + kOffBar;
  // barrier slots (8 bytes): a0_full[4] ae_full[4] a_empty[4] d_full[2] (+2 spare) d_free[2]; then the TMEM base pointer
  auto a0_full = [&](int c) { return bar0 + 8u * c; };
  auto ae_full = [&](int c) { return bar0 + 32u + 8u * c; };
  auto a_empty = [&](int c) { return bar0 + 64u + 8u * c; };
  auto d_full = [&](int d) { return bar0 + 96u + 8u * d; };
  auto d_free = [&](int d) { return bar0 + 128u + 8u * d; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar + 144);

  // ---- one-time setup ----------------------------------------------------------
  if (threadIdx.x == 0) {
    for (int c = 0; c < 4; ++c) {
      mbar_init(a0_full(c), 2 * kLoaderWarps * 32);   // every loader thread of both CTAs
      mbar_init(ae_full(c), 2 * kEpiWarps * 32);      // every epilogue thread of both CTAs
      mbar_init(a_empty(c), 1);
    }
    for (int d = 0; d < 4; ++d) mbar_init(d_full(d), 1);
    for (int d = 0; d < 2; ++d) mbar_init(d_free(d), 2 * kEpiWarps * 32);   // multi mode: accumulator drained
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  // resident B operands: scaled two-piece fp16 images of this CTA's 64 output features of every layer
  for (int l = 0; l < nl; ++l) {
    const float* W = p.W[l];
    const long long ldw = p.ldw[l];
    for (int item = threadIdx.x; item < 64 * 16; item += kThreads) {
      const int c = item & 15, nloc = item >> 4;      // 16-byte chunk = 8 k-values; local weight row
      const int n_glob = 64 * (int)rank + nloc;
      const float* src = W + (long long)n_glob * ldw + c * 8;
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(src));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
      uint32_t p1[4], p2[4];
      split2_scaled(v0.x, v0.y, kScaleW, p1[0], p2[0]);
      split2_scaled(v0.z, v0.w, kScaleW, p1[1], p2[1]);
      split2_scaled(v1.x, v1.y, kScaleW, p1[2], p2[2]);
      split2_scaled(v1.z, v1.w, kScaleW, p1[3], p2[3]);
      const int kb = c >> 3, cc = c & 7;
      uint8_t* img = sm + kOffW + l * kLayerBytes + kb * kImgBytes + (nloc >> 3) * 1024 + (nloc & 7) * 128 + ((cc ^ (nloc & 7)) << 4);
      *reinterpret_cast<uint4*>(img) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
      *reinterpret_cast<uint4*>(img + 2 * kImgBytes) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
    }
  }
  for (int i = threadIdx.x; i < kD; i += kThreads) {
    // hidden-layer biases are kept x kScaleA: their epilogue emits the next A operand already scaled
    for (int l = 0; l < kMaxLayers; ++l) s_const[l * kD + i] = (l < nl && p.bias[l]) ? __ldg(p.bias[l] + i) * ((l < nl - 1 && !kMulti) ? kScaleA : 1.f) : 0.f;
    if (kPre) s_const[2 * kD + i] = p.pre_bias ? __ldg(p.pre_bias + i) * kScaleA : 0.f;
    s_const[3 * kD + i] = has_dot ? __ldg(p.dot_w + i) : (has_ln ? __ldg(p.gamma + i) : 1.f);
    s_const[4 * kD + i] = has_ln ? __ldg(p.beta + i) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();            // both CTAs: barriers initialised, weights resident, TMEM allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const long long n_my = (p.num_tiles > pair) ? (p.num_tiles - pair + npairs - 1) / npairs : 0;

  if (warp < kLoaderWarps) {
    // ======================= loaders =======================
    reg_dec<kRegsLoader>();
    const int q = warp;
    const uint32_t buf0 = base + kOffLd + (uint32_t)(warp * kLoadBufs) * kChunkBytes;
    const int rl = lane >> 3, cj = lane & 7;          // copy domain: 8 lanes per 128-byte row piece
    const long long total = kPre ? 0 : n_my * 4;     // pre-stage mode: the epilogue builds the first operand
    const uint32_t a0_remote = map_to_leader(a0_full(0));   // the cluster window is linear: + 8 c
    Trace tr; tr.init(p, 2, warp == 0 && lane == 0);
    auto issue = [&](long long it, int b) {
      if (it < total) {
        const long long tile = pair + (it >> 2) * npairs;
        const int c = (int)(it & 3);
        const long long row0 = tile * kTileM + rank * 128 + q * 32;
        const uint32_t dst0 = buf0 + (uint32_t)b * kChunkBytes;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = i * 4 + rl;
          const long long row = row0 + r;
          const long long rc = row < p.M ? row : p.M - 1;
          cp_async16(dst0 + (uint32_t)(r * 128 + ((cj ^ (r & 7)) << 4)), p.A + rc * p.lda + c * 32 + cj * 4, row < p.M ? 16u : 0u);
        }
      }
      cp_async_commit();
    };
#pragma unroll
    for (int b = 0; b < kLoadBufs; ++b) issue(b, b);
    int b = 0;
    for (long long it = 0; it < total; ++it) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kLoadBufs - 1) : "memory");
      __syncwarp();
      const int c = (int)(it & 3);
      const uint32_t tph = (uint32_t)((it >> 2) & 1);
      tr.ev(0x60 + c);
      mbar_wait(a_empty(c), tph ^ 1u);              // last layer of the previous tile has read chunk c
      tc_fence_after();
      tr.ev(0x64 + c);
      const uint8_t* buf = sm + kOffLd + (warp * kLoadBufs + b) * kChunkBytes + lane * 128;
      const uint32_t ta = tmem_base + kTmemA + ((uint32_t)(q * 32) << 16) + (uint32_t)c * 16;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t p1[8], p2[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 x = *reinterpret_cast<const float4*>(buf + (((half * 4 + j) ^ (lane & 7)) << 4));
          split2_scaled(x.x, x.y, kScaleA, p1[2 * j], p2[2 * j]);
          split2_scaled(x.z, x.w, kScaleA, p1[2 * j + 1], p2[2 * j + 1]);
        }
        tmem_st8(ta + half * 8, p1);
        tmem_st8(ta + 64 + half * 8, p2);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive_remote(a0_remote + 8u * c);
      tr.ev(0x68 + c);
      __syncwarp();
      issue(it + kLoadBufs, b);
      b = (b + 1 == kLoadBufs) ? 0 : b + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp < kEpiWarp0) {
    // ======================= MMA issuer (leader CTA, warp 4, one thread) =======================
    reg_dec<kRegsMma>();
    if (rank == 0 && warp == kMmaWarp && lane == 0) {
      const uint64_t desc0 = make_desc(base + kOffW);
      Trace tr; tr.init(p, 0, true);
      uint32_t n_ae = 0;                            // completed phases of the ae_full barriers
      long long s = 0;                              // layer sequence number: accumulator = s & 1
#pragma unroll 1
      for (long long t = 0; t < n_my; ++t) {
#pragma unroll 1
        for (int l = 0; l < nl; ++l, ++s) {
          const uint64_t desc_l = desc0 + (uint64_t)((l * kLayerBytes) >> 4);
          const uint32_t d_tmem = tmem_base + kTmemD + (uint32_t)(s & 1) * kD;
          if (kMulti && s >= 2) {      // the products do not depend on each other: only the accumulator must be free
            mbar_wait(d_free((int)(s & 1)), (uint32_t)(((s >> 1) - 1) & 1));
            tc_fence_after();
          }
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            if (l == 0 && !kPre) mbar_wait(a0_full(c), (uint32_t)(t & 1));
            else if (!kMulti) mbar_wait(ae_full(c), n_ae & 1u);
            tc_fence_after();
            tr.ev(0x10 + l * 4 + c);
#pragma unroll
            for (int k2 = 0; k2 < 2; ++k2) {
              const int ks = 2 * c + k2;              // K = 16 step
              const uint32_t a1 = tmem_base + kTmemA + (uint32_t)ks * 8, a2 = a1 + 64;
              const uint64_t w1 = desc_l + (uint64_t)(((ks >> 2) * kImgBytes + (ks & 3) * 32) >> 4);
              const uint64_t w2 = w1 + (uint64_t)((2 * kImgBytes) >> 4);
              umma_f16_pair(d_tmem, a1, w2, kInstrDesc, ks != 0);       // smallest terms first
              umma_f16_pair(d_tmem, a2, w1, kInstrDesc, 1);
              umma_f16_pair(d_tmem, a1, w1, kInstrDesc, 1);
            }
            if (l == nl - 1) umma_commit_pair(a_empty(c));   // chunk c of the A operand may take the next tile
          }
          umma_commit_pair(d_full((int)(s & 1)));
          tr.ev(0x20 + l);
          if (l > 0 || kPre) ++n_ae;
        }
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    reg_inc<kRegsEpi>();
    const int ew = warp - kEpiWarp0;
    const int q = warp & 3, hf = ew >> 2;           // TMEM lane quarter, column half of every chunk
    uint8_t* slots = sm + kOffEp + ew * kEpiSlots * kSlotBytes;       // 4 tiles of 32 rows x 16 fp32
    float* xchg = reinterpret_cast<float*>(sm + kOffXchg);           // [2][8][32]
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int rl = lane >> 2, cc = lane & 3;        // coalesced domain: 4 lanes per 64-byte row piece, 8 rows per pass
    const bool has_add = has_g0 || has_g1;
    const uint32_t ae_remote = map_to_leader(ae_full(0));
    Trace tr; tr.init(p, ew == 0 ? 1 : 3, (ew == 0 || ew == 4) && lane == 0);
    // tile slot offset of (row r, 16-byte chunk ch): 64-byte rows, chunks rotated so that thread = row reads are conflict-free
    auto slot_off = [](int r, int ch) { return (uint32_t)(r * 64 + ((ch ^ ((r >> 1) & 3)) << 4)); };

    // Addend and residual rows are staged by this warp's own cp.async into its four 2 KB slots (no
    // registers, no scoreboard coupling).  Addends: step c uses slots 2 (c & 1) (gather0) and 2 (c & 1) + 1
    // (gather1), two steps in flight.  Residual: step c uses slot c, all four steps in flight from the end
    // of the first hidden layer; the slot just consumed doubles as the transpose tile of the output.
    // Row indices are loaded one tile ahead.
    const uint32_t slots_u = base + kOffEp + (uint32_t)ew * kEpiSlots * kSlotBytes;
    int ix0[4], ix1[4], ixr[4];                     // rows of gather0 / gather1 / residual for copy rows rl + 8 i
    int nx0[4], nx1[4], nxr[4];                     // the same for the next tile
    auto load_indices = [&](long long tile, int* a0, int* a1, int* ar) {
      const long long r0 = tile * kTileM + rank * 128 + q * 32;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        long long g = r0 + rl + 8 * i;
        g = g < p.M ? g : p.M - 1;
        a0[i] = (has_g0 && has_i0) ? __ldg(p.i0 + g) : (int)g;
        a1[i] = (has_g1 && has_i1) ? __ldg(p.i1 + g) : (int)g;
        ar[i] = (has_res && has_ridx) ? __ldg(p.res_idx + g) : (int)g;
      }
    };
    int pre_row = 0, pre_row_next = 0;              // pre-stage: this lane's row of the g2 table
    auto fetch_add = [&](int c) {
      const int col = 32 * c + 16 * hf + 4 * cc;
      const uint32_t dst = slots_u + (uint32_t)(2 * (c & 1)) * kSlotBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t off = slot_off(rl + 8 * i, cc);
        if (has_g0) cp_async16(dst + off, p.g0 + (long long)ix0[i] * p.ld_g0 + col, 16u);
        if (has_g1) cp_async16(dst + kSlotBytes + off, p.g1 + (long long)ix1[i] * p.ld_g1 + col, 16u);
      }
      cp_async_commit();
    };
    auto fetch_res = [&](int c) {                   // into slot c
      const int col = 32 * c + 16 * hf + 4 * cc;
      const uint32_t dst = slots_u + (uint32_t)c * kSlotBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async16(dst + slot_off(rl + 8 * i, cc), p.residual + (long long)ixr[i] * p.ld_res + col, 16u);
      cp_async_commit();
    };
    auto fetch_res_all = [&]() {
#pragma unroll
      for (int c = 0; c < 4; ++c) fetch_res(c);
    };
    auto first_fetch = [&]() {                      // what the tile needs first
      if (has_add) { fetch_add(0); fetch_add(1); }
      else if (has_res) fetch_res_all();
    };
    // thread = row read of this lane's 16 floats from a slot
    auto read_slot = [&](const uint8_t* slot, float* v) {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const float4 x = *reinterpret_cast<const float4*>(slot + slot_off(lane, ch));
        v[4 * ch] = x.x; v[4 * ch + 1] = x.y; v[4 * ch + 2] = x.z; v[4 * ch + 3] = x.w;
      }
    };
    // 16 accumulator columns -> A operand chunk c of the next layer.  The accumulator holds kScaleW * kScaleA
    // times the product and the next operand wants kScaleA times the activation:
    //   kScaleA * relu(acc / (kScaleW kScaleA) + b [+ ext]) = relu(acc / kScaleW + kScaleA b [+ kScaleA ext])
    // (exact power-of-two scalings; s_bias holds kScaleA * b, vc already includes kScaleA * ext).
    auto emit_chunk = [&](const float* vc, const float* s_bias, int c, bool has_ext, const float* ext) {
      const int col0 = 32 * c + 16 * hf;
      uint32_t p1[8], p2[8];
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        const float4 b4 = *reinterpret_cast<const float4*>(s_bias + col0 + 4 * j4);
        float y0 = fmaf(vc[4 * j4], 1.f / kScaleW, b4.x), y1 = fmaf(vc[4 * j4 + 1], 1.f / kScaleW, b4.y);
        float y2 = fmaf(vc[4 * j4 + 2], 1.f / kScaleW, b4.z), y3 = fmaf(vc[4 * j4 + 3], 1.f / kScaleW, b4.w);
        if (has_ext) {
          y0 = fmaf(ext[4 * j4], kScaleA, y0); y1 = fmaf(ext[4 * j4 + 1], kScaleA, y1);
          y2 = fmaf(ext[4 * j4 + 2], kScaleA, y2); y3 = fmaf(ext[4 * j4 + 3], kScaleA, y3);
        }
        split2(relu_nan(y0), relu_nan(y1), p1[2 * j4], p2[2 * j4]);
        split2(relu_nan(y2), relu_nan(y3), p1[2 * j4 + 1], p2[2 * j4 + 1]);
      }
      const uint32_t ta = lane_addr + kTmemA + (uint32_t)(16 * c + 8 * hf);
      tmem_st8(ta, p1);
      tmem_st8(ta + 64, p2);
      tr.ev(0x74);
      tmem_st_wait();
      tr.ev(0x75);
      tc_fence_before();
      mbar_arrive_remote(ae_remote + 8u * c);
    };

    auto load_pre_row = [&](long long tile) {
      long long g = tile * kTileM + rank * 128 + q * 32 + lane;
      g = g < p.M ? g : p.M - 1;
      return (int)__ldg(p.i2 + g);
    };
    if (n_my > 0) {
      load_indices(pair, ix0, ix1, ixr);
      if (kPre) pre_row = load_pre_row(pair);
      first_fetch();
    }
    long long s = 0;
#pragma unroll 1
    for (long long t = 0; t < n_my; ++t) {
      const long long tile = pair + t * npairs;
      const long long row0 = tile * kTileM + rank * 128 + q * 32;
      const bool tile_full = row0 + 32 <= p.M;      // warp-uniform: no per-row guards on the stores
      if (kMulti) {
        // ---- independent products: every accumulator goes straight to its own output
        const uint32_t dfree_remote = map_to_leader(d_free(0));
#pragma unroll 1
        for (int l = 0; l < nl; ++l, ++s) {
          mbar_wait(d_full((int)(s & 1)), (uint32_t)((s >> 1) & 1));
          tc_fence_after();
          const uint32_t d_addr = lane_addr + kTmemD + (uint32_t)(s & 1) * kD;
          float x[64];
#pragma unroll
          for (int c = 0; c < 4; ++c) tmem_ld16(d_addr + 32 * c + 16 * hf, x + 16 * c);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive_remote(dfree_remote + 8u * (uint32_t)(s & 1));     // accumulator drained
          const float* s_bias = s_const + l * kD;
          float* Yl = p.Ym[l];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint8_t* slot = slots + c * kSlotBytes;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 32 * c + 16 * hf + 4 * ch);
              *reinterpret_cast<float4*>(slot + slot_off(lane, ch)) =
                  make_float4(fmaf(x[16 * c + 4 * ch], kUnscaleD, b4.x), fmaf(x[16 * c + 4 * ch + 1], kUnscaleD, b4.y),
                              fmaf(x[16 * c + 4 * ch + 2], kUnscaleD, b4.z), fmaf(x[16 * c + 4 * ch + 3], kUnscaleD, b4.w));
            }
            __syncwarp();
            float4 o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = *reinterpret_cast<const float4*>(slot + slot_off(rl + 8 * i, cc));
            float* yrow = Yl + (row0 + rl) * p.ldy + 32 * c + 16 * hf + 4 * cc;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (tile_full || row0 + rl + 8 * i < p.M) stg_stream(reinterpret_cast<float4*>(yrow + (long long)(8 * i) * p.ldy), o[i]);
          }
          __syncwarp();
        }
        continue;
      }
      if (kPre) {
        // ---- pre-stage: first operand = relu(g2[i2] + g0[i0] + g1[i1] + bias), no accumulator involved
        const float* s_bias = s_const + 2 * kD;
        const float* trow = p.g2 + (long long)pre_row * p.ld_g2;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float ext[16];
          if (c < 3) asm volatile("cp.async.wait_group 1;" ::: "memory");
          else asm volatile("cp.async.wait_group 0;" ::: "memory");
          __syncwarp();
          const uint8_t* sp = slots + 2 * (c & 1) * kSlotBytes;
          read_slot(sp, ext);
          {
            float e1[16];
            read_slot(sp + kSlotBytes, e1);
#pragma unroll
            for (int j = 0; j < 16; ++j) ext[j] += e1[j];
          }
          __syncwarp();
          if (c + 2 < 4) fetch_add(c + 2);
          else if (c == 3 && has_res) fetch_res_all();
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 r4 = __ldg(reinterpret_cast<const float4*>(trow + 32 * c + 16 * hf + 4 * j4));
            ext[4 * j4] += r4.x; ext[4 * j4 + 1] += r4.y; ext[4 * j4 + 2] += r4.z; ext[4 * j4 + 3] += r4.w;
          }
          float zero[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) zero[j] = 0.f;
          mbar_wait(a_empty(c), (uint32_t)((t & 1) ^ 1));     // the previous tile's last layer has read chunk c
          tc_fence_after();
          emit_chunk(zero, s_bias, c, true, ext);
        }
      }
      // ---- hidden layers: accumulator -> bias (+ addends) -> ReLU -> split -> next A operand
#pragma unroll 1
      for (int l = 0; l < nl - 1; ++l, ++s) {
        const uint32_t d_addr = lane_addr + kTmemD + (uint32_t)(s & 1) * kD;
        const float* s_bias = s_const + l * kD;
        mbar_wait(d_full((int)(s & 1)), (uint32_t)((s >> 1) & 1));
        tc_fence_after();
        tr.ev(0x30 + l);
        if (l == 0 && has_add && !kPre) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float v[16];
            tmem_ld16(d_addr + 32 * c + 16 * hf, v);
            float ext[16];
            tr.ev(0x70);
            if (c < 3) asm volatile("cp.async.wait_group 1;" ::: "memory");   // steps c and c + 1 are in flight
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncwarp();
            tr.ev(0x71);
            const uint8_t* sp = slots + 2 * (c & 1) * kSlotBytes;
            if (has_g0) read_slot(sp, ext);
            if (has_g1) {
              float e1[16];
              read_slot(sp + kSlotBytes, e1);
#pragma unroll
              for (int j = 0; j < 16; ++j) ext[j] = has_g0 ? ext[j] + e1[j] : e1[j];
            }
            __syncwarp();
            if (c + 2 < 4) fetch_add(c + 2);
            else if (c == 3 && has_res) fetch_res_all();
            tr.ev(0x72);
            tmem_ld_wait();
            tr.ev(0x73);
            emit_chunk(v, s_bias, c, true, ext);
            tr.ev(0x40 + l * 4 + c);
          }
        } else {
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            float v[16];
            tmem_ld16(d_addr + 32 * c + 16 * hf, v);
            tmem_ld_wait();
            emit_chunk(v, s_bias, c, false, v);
            tr.ev(0x40 + l * 4 + c);
          }
        }
      }
      // ---- last layer
      {
        mbar_wait(d_full((int)(s & 1)), (uint32_t)((s >> 1) & 1));
        tc_fence_after();
        tr.ev(0x50);
        if (t + 1 < n_my) {                           // consumed at the end of this tile
          load_indices(tile + npairs, nx0, nx1, nxr);
          if (kPre) pre_row_next = load_pre_row(tile + npairs);
        }
        const uint32_t d_addr = lane_addr + kTmemD + (uint32_t)(s & 1) * kD;
        ++s;
        const float* s_bias = s_const + (nl - 1) * kD;
        float x[64];                                  // x[16 c + j] = column 32 c + 16 hf + j
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld16(d_addr + 32 * c + 16 * hf, x + 16 * c);
        tmem_ld_wait();
        tr.ev(0x51);
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 32 * c + 16 * hf + 4 * j4);
            x[16 * c + 4 * j4] = fmaf(x[16 * c + 4 * j4], kUnscaleD, b4.x);
            x[16 * c + 4 * j4 + 1] = fmaf(x[16 * c + 4 * j4 + 1], kUnscaleD, b4.y);
            x[16 * c + 4 * j4 + 2] = fmaf(x[16 * c + 4 * j4 + 2], kUnscaleD, b4.z);
            x[16 * c + 4 * j4 + 3] = fmaf(x[16 * c + 4 * j4 + 3], kUnscaleD, b4.w);
          }
        float* xa = xchg + (ew * 32 + lane);                        // slot 0: this warp's partials
        float* xb = xchg + (kEpiWarps * 32) + (ew * 32 + lane);     // slot 1
        const int partner = (ew ^ 4) * 32 + lane;
        if (has_dot) {
          // decoder tail: y = relu(x) . w + b, halves combined through smem (slot alternates per tile)
          float acc = 0.f;
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int j = 0; j < 16; ++j) acc = fmaf(relu_nan(x[16 * c + j]), s_const[3 * kD + 32 * c + 16 * hf + j], acc);
          float* mine = (t & 1) ? xb : xa;
          *mine = acc;
          named_bar_sync(1 + q, 64);
          if (hf == 0) {
            const float other = xchg[((t & 1) ? kEpiWarps * 32 : 0) + partner];
            const long long g = row0 + lane;
            if (g < p.M) p.Y[g * p.ldy] = acc + other + (p.dot_b ? __ldg(p.dot_b) : 0.f);
          }
        } else {
          if (has_ln) {
            // four independent partial sums: the reductions are dependency chains, not issue-bound
            float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
            for (int j = 0; j < 64; j += 4) { t0 += x[j]; t1 += x[j + 1]; t2 += x[j + 2]; t3 += x[j + 3]; }
            const float s1 = (t0 + t1) + (t2 + t3);
            *xa = s1;
            named_bar_sync(1 + q, 64);
            const float mu = (s1 + xchg[partner]) * (1.0f / kD);
            t0 = t1 = t2 = t3 = 0.f;
#pragma unroll
            for (int j = 0; j < 64; j += 4) {
              x[j] -= mu; x[j + 1] -= mu; x[j + 2] -= mu; x[j + 3] -= mu;
              t0 = fmaf(x[j], x[j], t0); t1 = fmaf(x[j + 1], x[j + 1], t1);
              t2 = fmaf(x[j + 2], x[j + 2], t2); t3 = fmaf(x[j + 3], x[j + 3], t3);
            }
            const float s2 = (t0 + t1) + (t2 + t3);
            *xb = s2;
            named_bar_sync(1 + q, 64);
            const float var = (s2 + xchg[kEpiWarps * 32 + partner]) * (1.0f / kD);
            const float rstd = 1.0f / sqrtf(var + p.eps);
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const int col = 32 * c + 16 * hf + 4 * j4;
                const float4 g4 = *reinterpret_cast<const float4*>(s_const + 3 * kD + col);
                const float4 e4 = *reinterpret_cast<const float4*>(s_const + 4 * kD + col);
                float* xx = x + 16 * c + 4 * j4;
                xx[0] = fmaf(xx[0] * rstd, g4.x, e4.x); xx[1] = fmaf(xx[1] * rstd, g4.y, e4.y);
                xx[2] = fmaf(xx[2] * rstd, g4.z, e4.z); xx[3] = fmaf(xx[3] * rstd, g4.w, e4.w);
              }
          }
          tr.ev(0x53);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint8_t* slot = slots + c * kSlotBytes;
            if (has_res) {
              // steps c .. 3 are in flight
              // (from step 2 on the next tile's first addend step may be pending behind them)
              const bool early = has_add && t + 1 < n_my;
              if (c == 0) asm volatile("cp.async.wait_group 3;" ::: "memory");
              else if (c == 1) asm volatile("cp.async.wait_group 2;" ::: "memory");
              else if (c == 2) { if (early) asm volatile("cp.async.wait_group 2;" ::: "memory"); else asm volatile("cp.async.wait_group 1;" ::: "memory"); }
              else { if (early) asm volatile("cp.async.wait_group 1;" ::: "memory"); else asm volatile("cp.async.wait_group 0;" ::: "memory"); }
              __syncwarp();
              float rsd[16];
              read_slot(slot, rsd);
#pragma unroll
              for (int j = 0; j < 16; ++j) x[16 * c + j] += rsd[j];
              __syncwarp();
            }
            // transpose through the same slot: thread = row writes, 4 lanes per row read and store 64 contiguous bytes
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
              *reinterpret_cast<float4*>(slot + slot_off(lane, ch)) =
                  make_float4(x[16 * c + 4 * ch], x[16 * c + 4 * ch + 1], x[16 * c + 4 * ch + 2], x[16 * c + 4 * ch + 3]);
            __syncwarp();
            float4 o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = *reinterpret_cast<const float4*>(slot + slot_off(rl + 8 * i, cc));
            float* yrow = p.Y + (row0 + rl) * p.ldy + 32 * c + 16 * hf + 4 * cc;
            if (tile_full) {
#pragma unroll
              for (int i = 0; i < 4; ++i) stg_stream(reinterpret_cast<float4*>(yrow + (long long)(8 * i) * p.ldy), o[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (row0 + rl + 8 * i < p.M) stg_stream(reinterpret_cast<float4*>(yrow + (long long)(8 * i) * p.ldy), o[i]);
            }
            __syncwarp();
            if (has_add && t + 1 < n_my && (c == 1 || c == 3)) {
              // slots 2 (c >> 1), 2 (c >> 1) + 1 are free again: the next tile's addend step c >> 1 can go now
              if (c == 1) {
#pragma unroll
                for (int i = 0; i < 4; ++i) { ix0[i] = nx0[i]; ix1[i] = nx1[i]; }
              }
              fetch_add(c >> 1);
            }
            tr.ev(0x54 + c);
          }
        }
      }
      tr.ev(0x52);
      if (t + 1 < n_my) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { ix0[i] = nx0[i]; ix1[i] = nx1[i]; ixr[i] = nxr[i]; }
        pre_row = pre_row_next;
        if (!(has_add && !has_dot)) first_fetch();      // with addends the two steps were issued inside the last layer
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }

  // ---- teardown ---------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();            // the peer may still be arriving on the leader's barriers
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

static unsigned long long* g_trace = nullptr;
static int g_trace_cap = 0;


// ---- two tiles in flight ----------------------------------------------------------------------------------
// The single-tile kernel above is bound by its epilogue warps: the MMA thread waits for them at every layer
// boundary and they wait for it.  With fp16 two-piece operands a tile needs 128 accumulator + 128 operand
// columns, so TWO tiles fit in tensor memory (slot S: D at 256 S, a1 | a2 at 256 S + 128) and every epilogue of
// one tile runs under the MMAs of the other:
//   MMA      : L0(X) L0(Y) | L1(X) L1(Y) | L2(X) L2(Y) | L0(X') ...
//   epilogue :       E0(X) | E0(Y) E1(X) | E1(Y) EL(X) | EL(Y) ...
// A tile has ONE accumulator: an epilogue first copies all of it to registers (64 values per thread) - its
// arrival for chunk 0 of the next operand (hidden layers) or on d_free (last layer) is what lets the next MMA of
// that slot overwrite it.  Specialised for the two block MLPs: 3 layers, gather0 (+ gather1), LayerNorm, residual
// by row (Spec<1>, Spec<2>).  All cp.async groups of a warp are consumed in the order they were issued, so one
// issued / consumed counter pair tells every wait how many younger groups may stay in flight.
__device__ __forceinline__ void cp_async_wait_pending(int n) {
  switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
  }
}

// Exact two-pass LayerNorm of a row held by two epilogue warps (this thread's 64 values in x): each pass publishes the
// half's sum in `mine`, meets the partner warp at named barrier 1 + q and adds the partner's `other`.  The partial
// sums t0..t3 over columns j = 0, 1, 2, 3 mod 4 run as two packed accumulators (t0, t1), (t2, t3) and are reduced as
// (t0 + t1) + (t2 + t3).
__device__ __forceinline__ float row_mean(const float* x, float* mine, const float* other, int q) {
  float2 ta = dup2(0.f), tb = dup2(0.f);
#pragma unroll
  for (int jj = 0; jj < 64; jj += 4) { ta = __fadd2_rn(ta, pair2(x + jj)); tb = __fadd2_rn(tb, pair2(x + jj + 2)); }
  const float s1 = (ta.x + ta.y) + (tb.x + tb.y);
  *mine = s1;
  named_bar_sync(1 + q, 64);
  return (s1 + *other) * (1.0f / kD);
}
// x -= mu in place; returns 1 / sqrt(var + eps)
__device__ __forceinline__ float row_rstd(float* x, float mu, float* mine, const float* other, int q, float eps) {
  float2 ta = dup2(0.f), tb = dup2(0.f);
#pragma unroll
  for (int jj = 0; jj < 64; jj += 4) {
    set2(x + jj, __fadd2_rn(pair2(x + jj), dup2(-mu)));
    set2(x + jj + 2, __fadd2_rn(pair2(x + jj + 2), dup2(-mu)));
    ta = __ffma2_rn(pair2(x + jj), pair2(x + jj), ta);
    tb = __ffma2_rn(pair2(x + jj + 2), pair2(x + jj + 2), tb);
  }
  const float s2 = (ta.x + ta.y) + (tb.x + tb.y);
  *mine = s2;
  named_bar_sync(1 + q, 64);
  const float var = (s2 + *other) * (1.0f / kD);
  return 1.0f / sqrtf(var + eps);
}
// x = (x rstd) gamma + beta, a multiply then an FMA; x[16 c + i] takes gamma[32 c + i], beta[32 c + i]
__device__ __forceinline__ void normalise(float* x, float rstd, const float* gamma, const float* beta) {
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
      const float4 g4 = *reinterpret_cast<const float4*>(gamma + 32 * c + 4 * j4);
      const float4 e4 = *reinterpret_cast<const float4*>(beta + 32 * c + 4 * j4);
      float* xx = x + 16 * c + 4 * j4;
      set2(xx, __ffma2_rn(__fmul2_rn(pair2(xx), dup2(rstd)), make_float2(g4.x, g4.y), make_float2(e4.x, e4.y)));
      set2(xx + 2, __ffma2_rn(__fmul2_rn(pair2(xx + 2), dup2(rstd)), make_float2(g4.z, g4.w), make_float2(e4.z, e4.w)));
    }
}

template <int SPEC, bool STASH = false, bool PSUM = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) tc_chain2_kernel(const Params p) {
  // STASH (training forward): the hidden ReLU outputs, the LayerNorm input and the row statistics are written out as well
  static_assert(!STASH || !Spec<SPEC>::pre, "the stash belongs to the three-layer forms");
  // Rows may be paired destination slots (p.edge_slots): a negative gather index i0 marks a padding slot, whose gathers
  // read row 0 and whose output row is +0.0.  PSUM: the store emits node rows (0 + y[2v]) + y[2v + 1] instead of y -
  // slots 2v, 2v + 1 are adjacent rows of the transpose tile, so the pair sum is formed where the stores are.
  static_assert(!PSUM || !STASH, "the pair-sum output is an inference form");
  // kPre (Spec<7>): the first operand is built by the epilogue warps from three gathers (no loader, two MMA layers,
  // residual through a small table read directly); otherwise three MMA layers, residual rows = the tile's rows.
  constexpr bool kPre = Spec<SPEC>::pre;
  static_assert(Spec<SPEC>::g0 == 1 && Spec<SPEC>::res == 1 && Spec<SPEC>::ln == 1 && Spec<SPEC>::dot == 0 &&
                ((kPre && Spec<SPEC>::nl == 2 && Spec<SPEC>::ridx == 1) || (!kPre && Spec<SPEC>::nl == 3 && Spec<SPEC>::ridx == 0)),
                "two-tile form: addends, LayerNorm, residual; 3 layers, or pre-stage + 2 layers");
  constexpr int nl = Spec<SPEC>::nl;
  // the pre-stage form has no loader work (the epilogue builds the first operand): its registers go to the epilogue
  constexpr int kRegsLd = kPre ? 56 : kRegsLoader, kRegsEp = kPre ? 208 : kRegsEpi;
  static_assert(32 * (4 * kRegsLd + 4 * kRegsMma + kEpiWarps * kRegsEp) <= kThreads * 128, "setmaxnreg budget");
  constexpr bool has_i0 = Spec<SPEC>::i0 != 0, has_g1 = Spec<SPEC>::g1 != 0, has_i1 = Spec<SPEC>::i1 != 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  float* s_const = reinterpret_cast<float*>(sm + kOffConst);   // bias[0..2] (hidden ones x kScaleA), gamma, beta
  const uint32_t bar0 = base + kOffBar;
  // per slot S (112 bytes): a0_full[4] ae_full[4] a_empty[4] d_full d_free; then the TMEM base pointer
  auto a0_full = [&](int S, int c) { return bar0 + 112u * S + 8u * c; };
  auto ae_full = [&](int S, int c) { return bar0 + 112u * S + 32u + 8u * c; };
  auto a_empty = [&](int S, int c) { return bar0 + 112u * S + 64u + 8u * c; };
  auto d_full = [&](int S) { return bar0 + 112u * S + 96u; };
  auto d_free = [&](int S) { return bar0 + 112u * S + 104u; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar + 224);

  if (threadIdx.x == 0) {
    for (int S = 0; S < 2; ++S) {
      for (int c = 0; c < 4; ++c) {
        mbar_init(a0_full(S, c), 2 * kLoaderWarps * 32);
        mbar_init(ae_full(S, c), 2 * kEpiWarps * 32);
        mbar_init(a_empty(S, c), 1);
      }
      mbar_init(d_full(S), 1);
      mbar_init(d_free(S), 2 * kEpiWarps * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int l = 0; l < nl; ++l) {
    const float* W = p.W[l];
    const long long ldw = p.ldw[l];
    for (int item = threadIdx.x; item < 64 * 16; item += kThreads) {
      const int c = item & 15, nloc = item >> 4;
      const float* src = W + (long long)(64 * (int)rank + nloc) * ldw + c * 8;
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(src));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
      uint32_t p1[4], p2[4];
      split2_scaled(v0.x, v0.y, kScaleW, p1[0], p2[0]);
      split2_scaled(v0.z, v0.w, kScaleW, p1[1], p2[1]);
      split2_scaled(v1.x, v1.y, kScaleW, p1[2], p2[2]);
      split2_scaled(v1.z, v1.w, kScaleW, p1[3], p2[3]);
      const int kb = c >> 3, cc = c & 7;
      uint8_t* img = sm + kOffW + l * kLayerBytes + kb * kImgBytes + (nloc >> 3) * 1024 + (nloc & 7) * 128 + ((cc ^ (nloc & 7)) << 4);
      *reinterpret_cast<uint4*>(img) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
      *reinterpret_cast<uint4*>(img + 2 * kImgBytes) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
    }
  }
  for (int i = threadIdx.x; i < kD; i += kThreads) {
    for (int l = 0; l < nl; ++l) s_const[l * kD + i] = p.bias[l] ? __ldg(p.bias[l] + i) * (l < nl - 1 ? kScaleA : 1.f) : 0.f;
    if (kPre) s_const[2 * kD + i] = p.pre_bias ? __ldg(p.pre_bias + i) * kScaleA : 0.f;
    s_const[3 * kD + i] = __ldg(p.gamma + i);
    s_const[4 * kD + i] = __ldg(p.beta + i);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const long long n_my = (p.num_tiles > pair) ? (p.num_tiles - pair + npairs - 1) / npairs : 0;   // tile j -> slot j & 1

  if (warp < kLoaderWarps) {
    // ======================= loaders =======================
    reg_dec<kRegsLd>();
    const int q = warp;
    const uint32_t buf0 = base + kOffLd + (uint32_t)(warp * kLoadBufs) * kChunkBytes;
    const int rl = lane >> 3, cj = lane & 7;
    const long long total = kPre ? 0 : n_my * 4;
    const uint32_t a0_remote = map_to_leader(a0_full(0, 0));
    const uint64_t pol_keep = l2_policy_evict_last();
    auto issue = [&](long long it, int b) {
      if (it < total) {
        const long long tile = pair + (it >> 2) * npairs;
        const int c = (int)(it & 3);
        const long long row0 = tile * kTileM + rank * 128 + q * 32;
        const uint32_t dst0 = buf0 + (uint32_t)b * kChunkBytes;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = i * 4 + rl;
          const long long row = row0 + r;
          const long long rc = row < p.M ? row : p.M - 1;
          cp_async16_hint(dst0 + (uint32_t)(r * 128 + ((cj ^ (r & 7)) << 4)), p.A + rc * p.lda + c * 32 + cj * 4, row < p.M ? 16u : 0u, pol_keep);
        }
      }
      cp_async_commit();
    };
#pragma unroll
    for (int b = 0; b < kLoadBufs; ++b) issue(b, b);
    int b = 0;
    for (long long it = 0; it < total; ++it) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kLoadBufs - 1) : "memory");
      __syncwarp();
      const int c = (int)(it & 3);
      const long long j = it >> 2;
      const int S = (int)(j & 1);
      mbar_wait(a_empty(S, c), (uint32_t)(((j >> 1) & 1) ^ 1));   // the slot's previous tile has read chunk c
      tc_fence_after();
      const uint8_t* buf = sm + kOffLd + (warp * kLoadBufs + b) * kChunkBytes + lane * 128;
      const uint32_t ta = tmem_base + (uint32_t)S * 256 + 128 + ((uint32_t)(q * 32) << 16) + (uint32_t)c * 16;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t p1[8], p2[8];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const float4 x = *reinterpret_cast<const float4*>(buf + (((half * 4 + jj) ^ (lane & 7)) << 4));
          split2_scaled(x.x, x.y, kScaleA, p1[2 * jj], p2[2 * jj]);
          split2_scaled(x.z, x.w, kScaleA, p1[2 * jj + 1], p2[2 * jj + 1]);
        }
        tmem_st8(ta + half * 8, p1);
        tmem_st8(ta + 64 + half * 8, p2);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive_remote(a0_remote + 112u * (uint32_t)S + 8u * (uint32_t)c);
      __syncwarp();
      issue(it + kLoadBufs, b);
      b = (b + 1 == kLoadBufs) ? 0 : b + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp < kEpiWarp0) {
    // ======================= MMA issuer =======================
    reg_dec<kRegsMma>();
    if (rank == 0 && warp == kMmaWarp && lane == 0) {
      const uint64_t desc0 = make_desc(base + kOffW);
      const long long groups = (n_my + 1) >> 1;
#pragma unroll 1
      for (long long g = 0; g < groups; ++g) {
#pragma unroll 1
        for (int l = 0; l < nl; ++l) {
          const uint64_t desc_l = desc0 + (uint64_t)((l * kLayerBytes) >> 4);
#pragma unroll 1
          for (int S = 0; S < 2; ++S) {
            if (2 * g + S >= n_my) continue;
            const uint32_t d_tmem = tmem_base + (uint32_t)S * 256;
            const uint32_t a_base = d_tmem + 128;
            if (l == 0 && g > 0) {                  // the slot's previous tile has copied its last accumulator out
              mbar_wait(d_free(S), (uint32_t)((g - 1) & 1));
              tc_fence_after();
            }
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
              // the slot's ae_full barriers complete (nl - 1) times per tile: phase index g (nl - 1) + (l - 1)
              // (both forms complete a slot's ae_full barriers twice per tile)
              if (!kPre && l == 0) mbar_wait(a0_full(S, c), (uint32_t)(g & 1));
              else mbar_wait(ae_full(S, c), (uint32_t)((g * 2 + (kPre ? l : l - 1)) & 1));
              tc_fence_after();
#pragma unroll
              for (int k2 = 0; k2 < 2; ++k2) {
                const int ks = 2 * c + k2;
                const uint32_t a1 = a_base + (uint32_t)ks * 8, a2 = a1 + 64;
                const uint64_t w1 = desc_l + (uint64_t)(((ks >> 2) * kImgBytes + (ks & 3) * 32) >> 4);
                const uint64_t w2 = w1 + (uint64_t)((2 * kImgBytes) >> 4);
                umma_f16_pair(d_tmem, a1, w2, kInstrDesc, ks != 0);
                umma_f16_pair(d_tmem, a2, w1, kInstrDesc, 1);
                umma_f16_pair(d_tmem, a1, w1, kInstrDesc, 1);
              }
              if (l == nl - 1) umma_commit_pair(a_empty(S, c));
            }
            umma_commit_pair(d_full(S));
          }
        }
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    reg_inc<kRegsEp>();
    const int ew = warp - kEpiWarp0;
    const int q = warp & 3, hf = ew >> 2;
    uint8_t* slots = sm + kOffEp + ew * kEpiSlots * kSlotBytes;
    const uint32_t slots_u = base + kOffEp + (uint32_t)ew * kEpiSlots * kSlotBytes;
    float* xchg = reinterpret_cast<float*>(sm + kOffXchg);
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int rl = lane >> 2, cc = lane & 3;
    const uint32_t ae_remote = map_to_leader(ae_full(0, 0)), dfree_remote = map_to_leader(d_free(0));
    auto slot_off = [](int r, int ch) { return (uint32_t)(r * 64 + ((ch ^ ((r >> 1) & 3)) << 4)); };
    auto read_slot = [&](const uint8_t* slot, float* v) {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const float4 x = *reinterpret_cast<const float4*>(slot + slot_off(lane, ch));
        v[4 * ch] = x.x; v[4 * ch + 1] = x.y; v[4 * ch + 2] = x.z; v[4 * ch + 3] = x.w;
      }
    };
    auto tile_row0 = [&](long long j) { return (pair + j * npairs) * kTileM + rank * 128 + q * 32; };

    // ---- the cp.async stream (FIFO: consumed in issue order) ----
    int issued = 0, consumed = 0;
    auto wait_next = [&]() { cp_async_wait_pending(issued - consumed - 1); ++consumed; };
    // Row pointers (lane's 16-byte column piece included) are formed once per tile: a step then costs one
    // cp.async per row with the step's column offset as an immediate.
    const float* pr0[4]; const float* pr1[4];       // gather rows of the tile whose addend steps are being issued
    const float* nr0[4]; const float* nr1[4];       // ... of the tile after it
    const float* pres[4];                           // residual rows of the tile whose residual steps are being issued
    uint32_t soff[4];                               // this lane's destinations inside a slot
#pragma unroll
    for (int i = 0; i < 4; ++i) soff[i] = slot_off(rl + 8 * i, cc);
    const int lane_col = 16 * hf + 4 * cc;
    const uint64_t pol_drop = l2_policy_evict_first();
    auto load_indices = [&](long long j, const float** a0, const float** a1) {
      const long long r0 = tile_row0(j);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        long long g = r0 + rl + 8 * i;
        g = g < p.M ? g : p.M - 1;
        a0[i] = p.g0 + (has_i0 ? (long long)max(__ldg(p.i0 + g), 0) : g) * p.ld_g0 + lane_col;
        if (has_g1) a1[i] = p.g1 + (has_i1 ? (long long)__ldg(p.i1 + g) : g) * p.ld_g1 + lane_col;
      }
    };
    auto res_rows = [&](long long j) {
      const long long r0 = tile_row0(j);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        long long g = r0 + rl + 8 * i;
        g = g < p.M ? g : p.M - 1;
        pres[i] = p.residual + g * p.ld_res + lane_col;
      }
    };
    long long add_k = 0;                            // addend steps issued so far (step k -> slots 2 (k & 1), + 1)
    auto fetch_add = [&](int c) {                   // step c of the tile pr0 / pr1 describe
      const uint32_t dst = slots_u + (uint32_t)(2 * (add_k & 1)) * kSlotBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        cp_async16(dst + soff[i], pr0[i] + 32 * c, 16u);
        if (has_g1) cp_async16(dst + kSlotBytes + soff[i], pr1[i] + 32 * c, 16u);
      }
      cp_async_commit();
      ++issued; ++add_k;
    };
    auto fetch_res = [&](int c) {                   // step c of the tile pres describes -> slot c
      const uint32_t dst = slots_u + (uint32_t)c * kSlotBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async16_hint(dst + soff[i], pres[i] + 32 * c, 16u, pol_drop);
      cp_async_commit();
      ++issued;
    };
    // `strow` (STASH): where this thread's row of the activation being emitted is kept for the backward pass (NULL past M)
    auto emit_chunk = [&](const float* vc, const float* s_bias, int S, int c, const float* ext, bool has_ext, float* strow) {
      const int col0 = 32 * c + 16 * hf;
      uint32_t p1[8], p2[8];
      float st[STASH ? 16 : 1];
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        const float4 b4 = *reinterpret_cast<const float4*>(s_bias + col0 + 4 * j4);
        float2 ya = __ffma2_rn(pair2(vc + 4 * j4), dup2(1.f / kScaleW), make_float2(b4.x, b4.y));
        float2 yb = __ffma2_rn(pair2(vc + 4 * j4 + 2), dup2(1.f / kScaleW), make_float2(b4.z, b4.w));
        if (has_ext) {
          ya = __ffma2_rn(pair2(ext + 4 * j4), dup2(kScaleA), ya);
          yb = __ffma2_rn(pair2(ext + 4 * j4 + 2), dup2(kScaleA), yb);
        }
        ya.x = relu_nan(ya.x); ya.y = relu_nan(ya.y); yb.x = relu_nan(yb.x); yb.y = relu_nan(yb.y);
        if (STASH) {                                // exact: kScaleA is a power of two
          set2(st + 4 * j4, __fmul2_rn(ya, dup2(1.f / kScaleA)));
          set2(st + 4 * j4 + 2, __fmul2_rn(yb, dup2(1.f / kScaleA)));
        }
        split2(ya, p1[2 * j4], p2[2 * j4]);
        split2(yb, p1[2 * j4 + 1], p2[2 * j4 + 1]);
      }
      if (STASH && strow) { stg256(strow + col0, st); stg256(strow + col0 + 8, st + 8); }
      const uint32_t ta = lane_addr + (uint32_t)S * 256 + 128 + (uint32_t)(16 * c + 8 * hf);
      tmem_st8(ta, p1);
      tmem_st8(ta + 64, p2);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive_remote(ae_remote + 112u * (uint32_t)S + 8u * (uint32_t)c);
    };

    uint32_t dcnt0 = 0, dcnt1 = 0;                  // d_full phases consumed per slot
    auto wait_acc = [&](int S, float* v) {          // the slot's accumulator -> 64 registers
      mbar_wait(d_full(S), (S ? dcnt1 : dcnt0) & 1u);
      if (S) ++dcnt1; else ++dcnt0;
      tc_fence_after();
      const uint32_t d_addr = lane_addr + (uint32_t)S * 256;
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld16(d_addr + 32 * c + 16 * hf, v + 16 * c);
      tmem_ld_wait();
    };

    const long long groups = (n_my + 1) >> 1;
    if (n_my > 0) {
      load_indices(0, pr0, pr1);
      fetch_add(0); fetch_add(1);
      if (n_my > 1) load_indices(1, nr0, nr1);
    }
#pragma unroll 1
    for (long long g = 0; g < groups; ++g) {
      const long long jX = 2 * g, jY = 2 * g + 1;
      const bool hasY = jY < n_my, hasNext = jY + 1 < n_my;
      // ---- addend stage (E0, or the pre-stage that builds the first operand): addends + bias + ReLU -> operand
#pragma unroll 1
      for (int S = 0; S < 2; ++S) {
        if (S == 1 && !hasY) break;
        float v[64];
        const float* trow = nullptr;
        float* st1 = nullptr;
        if (STASH) {
          const long long gr = tile_row0(2 * g + S) + lane;
          if (gr < p.M) st1 = p.st_a1 + gr * p.ld_st;
        }
        if (kPre) {
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] = 0.f;
          long long gr = tile_row0(2 * g + S) + lane;
          gr = gr < p.M ? gr : p.M - 1;
          trow = p.g2 + (long long)__ldg(p.i2 + gr) * p.ld_g2 + 16 * hf;
        } else {
          wait_acc(S, v);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float ext[16];
          wait_next();
          __syncwarp();
          const uint8_t* sp = slots + 2 * (c & 1) * kSlotBytes;      // add_k parity == c parity (4 steps per tile)
          read_slot(sp, ext);
          if (has_g1) {
            float e1[16];
            read_slot(sp + kSlotBytes, e1);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) set2(ext + jj, __fadd2_rn(pair2(ext + jj), pair2(e1 + jj)));
          }
          __syncwarp();
          // next issue of the stream: two addend steps stay in flight; after a tile's last two steps the
          // stream moves to the next tile's addends, or (after the group's last tile) to the residuals of X
          if (c < 2) {
            fetch_add(c + 2);
            if (c == 1) {                           // this tile's steps are all issued: indices of the next tile
#pragma unroll
              for (int i = 0; i < 4; ++i) { pr0[i] = nr0[i]; if (has_g1) pr1[i] = nr1[i]; }
            }
          } else if (S == 0 && hasY) {
            fetch_add(c - 2);                       // addends of Y, steps 0 and 1
          } else if (!kPre) {                       // last tile of the group: residual steps of X (slots 2(c-2), +1 are free)
            if (c == 2) res_rows(jX);
            fetch_res(2 * (c - 2));
            fetch_res(2 * (c - 2) + 1);
          }
          if (kPre) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 r4 = __ldg(reinterpret_cast<const float4*>(trow + 32 * c + 4 * j4));
              set2(ext + 4 * j4, __fadd2_rn(pair2(ext + 4 * j4), make_float2(r4.x, r4.y)));
              set2(ext + 4 * j4 + 2, __fadd2_rn(pair2(ext + 4 * j4 + 2), make_float2(r4.z, r4.w)));
            }
            mbar_wait(a_empty(S, c), (uint32_t)((g & 1) ^ 1));      // the slot's previous tile has read chunk c
            tc_fence_after();
          }
          emit_chunk(v + 16 * c, s_const + (kPre ? 2 * kD : 0), S, c, ext, true, st1);
        }
      }
      // all addend steps of this group are issued: gather rows of the next group's tiles (X' straight into the
      // live set - its first steps are issued inside this group's last layer -, Y' into the spare set)
      if (hasNext) load_indices(jY + 1, pr0, pr1);
      if (jY + 2 < n_my) load_indices(jY + 2, nr0, nr1);
      // ---- E1: bias + ReLU -> next operand
#pragma unroll 1
      for (int S = 0; S < 2; ++S) {
        if (S == 1 && !hasY) break;
        float v[64];
        float* st2 = nullptr;
        if (STASH) {
          const long long gr = tile_row0(2 * g + S) + lane;
          if (gr < p.M) st2 = p.st_a2 + gr * p.ld_st;
        }
        wait_acc(S, v);
#pragma unroll
        for (int c = 0; c < 4; ++c) emit_chunk(v + 16 * c, s_const + (kPre ? 0 : kD), S, c, v, false, st2);
      }
      // ---- last layer: LayerNorm + residual + store
#pragma unroll 1
      for (int S = 0; S < 2; ++S) {
        if (S == 1 && !hasY) break;
        const long long row0 = tile_row0(2 * g + S);
        const bool tile_full = row0 + 32 <= p.M;
        const bool pad_row = has_i0 && p.edge_slots && row0 + lane < p.M && __ldg(p.i0 + row0 + lane) < 0;
        if (!kPre && S == 0 && hasY) res_rows(jY);    // X's residual steps are all issued: the stream continues with Y's
        const float* rrow = nullptr;
        if (kPre) {
          long long gr = row0 + lane;
          gr = gr < p.M ? gr : p.M - 1;
          rrow = p.residual + (long long)__ldg(p.res_idx + gr) * p.ld_res + 16 * hf;
        }
        float x[64];
        wait_acc(S, x);
        tc_fence_before();
        mbar_arrive_remote(dfree_remote + 112u * (uint32_t)S);      // accumulator copied out
        const float* s_bias = s_const + (nl - 1) * kD;
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 32 * c + 16 * hf + 4 * j4);
            float* xx = x + 16 * c + 4 * j4;
            set2(xx, __ffma2_rn(pair2(xx), dup2(kUnscaleD), make_float2(b4.x, b4.y)));
            set2(xx + 2, __ffma2_rn(pair2(xx + 2), dup2(kUnscaleD), make_float2(b4.z, b4.w)));
          }
        const bool st_row = STASH && row0 + lane < p.M;
        if (STASH && st_row) {                                      // the LayerNorm input, as the backward reads it
          float* zr = p.st_z + (row0 + lane) * p.ld_st + 16 * hf;
#pragma unroll
          for (int c = 0; c < 4; ++c) { stg256(zr + 32 * c, x + 16 * c); stg256(zr + 32 * c + 8, x + 16 * c + 8); }
        }
        float* xa = xchg + (ew * 32 + lane);
        float* xb = xchg + (kEpiWarps * 32) + (ew * 32 + lane);
        const int partner = (ew ^ 4) * 32 + lane;
        const float mu = row_mean(x, xa, xchg + partner, q);
        const float rstd = row_rstd(x, mu, xb, xchg + kEpiWarps * 32 + partner, q, p.eps);
        if (STASH && st_row && hf == 0) { p.st_mean[row0 + lane] = mu; p.st_rstd[row0 + lane] = rstd; }
        normalise(x, rstd, s_const + 3 * kD + 16 * hf, s_const + 4 * kD + 16 * hf);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint8_t* slot = slots + c * kSlotBytes;
          if (kPre) {                                               // residual through a small table: direct reads
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 r4 = __ldg(reinterpret_cast<const float4*>(rrow + 32 * c + 4 * j4));
              float* xx = x + 16 * c + 4 * j4;
              set2(xx, __fadd2_rn(pair2(xx), make_float2(r4.x, r4.y)));
              set2(xx + 2, __fadd2_rn(pair2(xx + 2), make_float2(r4.z, r4.w)));
            }
          } else {
            wait_next();                                            // residual step c of this tile
            __syncwarp();
            float rsd[16];
            read_slot(slot, rsd);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) set2(x + 16 * c + jj, __fadd2_rn(pair2(x + 16 * c + jj), pair2(rsd + jj)));
            __syncwarp();
          }
          if (pad_row) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) x[16 * c + jj] = 0.f;
          }
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
            *reinterpret_cast<float4*>(slot + slot_off(lane, ch)) =
                make_float4(x[16 * c + 4 * ch], x[16 * c + 4 * ch + 1], x[16 * c + 4 * ch + 2], x[16 * c + 4 * ch + 3]);
          __syncwarp();
          if (PSUM) {                                               // node rows row0 / 2 + rl (+ 8): slot rows 2 rl, 2 rl + 1 (+ 16)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const int nr = rl + 8 * k;
              const float4 a = *reinterpret_cast<const float4*>(slot + slot_off(2 * nr, cc));
              const float4 b = *reinterpret_cast<const float4*>(slot + slot_off(2 * nr + 1, cc));
              const float2 o01 = __fadd2_rn(__fadd2_rn(dup2(0.f), make_float2(a.x, a.y)), make_float2(b.x, b.y));
              const float2 o23 = __fadd2_rn(__fadd2_rn(dup2(0.f), make_float2(a.z, a.w)), make_float2(b.z, b.w));
              const float4 o = make_float4(o01.x, o01.y, o23.x, o23.y);
              if (tile_full || row0 + 2 * nr < p.M)
                stg_hint(reinterpret_cast<float4*>(p.Y + ((row0 >> 1) + nr) * p.ldy + 32 * c + 16 * hf + 4 * cc), o, pol_drop);
            }
          } else {
            float4 o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = *reinterpret_cast<const float4*>(slot + slot_off(rl + 8 * i, cc));
            float* yrow = p.Y + (row0 + rl) * p.ldy + 32 * c + 16 * hf + 4 * cc;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (tile_full || row0 + rl + 8 * i < p.M) stg_hint(reinterpret_cast<float4*>(yrow + (long long)(8 * i) * p.ldy), o[i], pol_drop);
          }
          __syncwarp();
          // the slot is free again: next group of the stream
          if (!kPre && S == 0 && hasY) fetch_res(c);                // residual of Y, step c
          else if ((S == 1 || !hasY) && hasNext && (c == 1 || c == 3)) fetch_add(c >> 1);   // slots free: next group's X, step c >> 1
        }
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}


// ---- two tiles in flight, shapes without gathered addends -------------------------------------------------------
// NL layers (2 or 3); K2: the first layer contracts two operands (z0 = A W0^T + A2 W_A2^T + b0, the node processor's
// cat([x, agg]) @ V0^T of models/GNN.py:100 - no intermediate T = x Va^T tensor, no addend stage: the loader writes
// the second operand into the same TMEM chunks once the first operand's MMAs have read them); RES: residual = the
// tile's own rows of p.residual; TAIL 0: LayerNorm (if gamma) + residual -> Y, TAIL 1: relu . dot_w + dot_b.
// Shared memory: (NL + K2) weight images, loader ring, two 2 KB slots per epilogue warp (residual ring / transpose).
template <int NL, bool K2, bool RES, int TAIL, bool SYN = false, bool AGG = false, bool PAIR = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) tc_chain2n_kernel(const Params p) {
  static_assert(!(SYN && K2), "the synthesised operand is a single-operand form");
  // AGG: the first operand is not read but FORMED by the loader - row m = e[eid0] + e[eid1], the destination-ordered sum of
  // the (at most two) edge rows arriving at node m (scatter_sum, models/GNN.py:99, for in-degree <= 2: (0 + a) + b is the
  // reference's order bit for bit).  The aggregation launch, its [N, 128] result and the re-read of it disappear: every
  // edge row is read once, here.  Source 0 rides the cp.async ring (row addresses through the index), source 1 comes as
  // four 256-bit loads per chunk in the thread = row layout the ring is read back in.
  static_assert(!AGG || (K2 && NL == 3 && RES && TAIL == 0 && !SYN), "AGG belongs to the two-operand node form");
  // PAIR (an AGG form): A is the paired destination slot table (gnc_grid_pair_slots) and row m's edge rows are the adjacent
  // rows 2m, 2m + 1 (a zero row where an edge is missing) - the same two sources, with addresses instead of index lookups.
  static_assert(!PAIR || AGG, "PAIR is a form of AGG");
  // loaders that form their operand (AGG, PAIR, SYN) take registers from the epilogue: the smallest splits without spills
  constexpr int kRegsLd = PAIR ? 96 : (AGG || SYN) ? 88 : kRegsLoader, kRegsEp = PAIR ? 184 : (AGG || SYN) ? 192 : kRegsEpi;
  static_assert(32 * (4 * kRegsLd + 4 * kRegsMma + kEpiWarps * kRegsEp) <= kThreads * 128, "setmaxnreg budget");
  constexpr int kImgs = NL + (K2 ? 1 : 0);
  static_assert(kImgs <= 4 && NL >= 2, "at most four weight images");
  constexpr int kOffLd2 = kImgs * kLayerBytes;
  constexpr int kOffEp2 = kOffLd2 + kLoaderWarps * kLoadBufs * kChunkBytes;
  constexpr int kOffConst2 = kOffEp2 + kEpiWarps * 2 * kSlotBytes;
  constexpr int kOffXchg2 = kOffConst2 + 5 * kD * 4;
  constexpr int kOffBar2 = kOffXchg2 + 2 * kEpiWarps * 32 * 4;
  static_assert(kOffBar2 + 320 + 1024 <= 232448, "shared memory layout");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  float* s_const = reinterpret_cast<float*>(sm + kOffConst2);
  const uint32_t bar0 = base + kOffBar2;
  // per slot S (144 bytes): a0_full[4] ae_full[4] a_empty[4] a_mid[4] d_full d_free; then the TMEM base pointer
  auto a0_full = [&](int S, int c) { return bar0 + 144u * S + 8u * c; };
  auto ae_full = [&](int S, int c) { return bar0 + 144u * S + 32u + 8u * c; };
  auto a_empty = [&](int S, int c) { return bar0 + 144u * S + 64u + 8u * c; };
  auto a_mid = [&](int S, int c) { return bar0 + 144u * S + 96u + 8u * c; };
  auto d_full = [&](int S) { return bar0 + 144u * S + 128u; };
  auto d_free = [&](int S) { return bar0 + 144u * S + 136u; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar2 + 288);

  if (threadIdx.x == 0) {
    for (int S = 0; S < 2; ++S) {
      for (int c = 0; c < 4; ++c) {
        mbar_init(a0_full(S, c), 2 * kLoaderWarps * 32);
        mbar_init(ae_full(S, c), 2 * kEpiWarps * 32);
        mbar_init(a_empty(S, c), 1);
        mbar_init(a_mid(S, c), 1);
      }
      mbar_init(d_full(S), 1);
      mbar_init(d_free(S), 2 * kEpiWarps * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  // weight images: [W[0]] [W_A2 if K2] [W[1]] ... [W[NL-1]]
  for (int im = 0; im < kImgs; ++im) {
    const int l = (K2 && im >= 1) ? im - 1 : im;
    const float* W = (K2 && im == 1) ? p.W_A2 : p.W[l];
    const long long ldw = (K2 && im == 1) ? p.ldw_A2 : p.ldw[l];
    for (int item = threadIdx.x; item < 64 * 16; item += kThreads) {
      const int c = item & 15, nloc = item >> 4;
      const float* src = W + (long long)(64 * (int)rank + nloc) * ldw + c * 8;
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(src));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
      uint32_t p1[4], p2[4];
      split2_scaled(v0.x, v0.y, kScaleW, p1[0], p2[0]);
      split2_scaled(v0.z, v0.w, kScaleW, p1[1], p2[1]);
      split2_scaled(v1.x, v1.y, kScaleW, p1[2], p2[2]);
      split2_scaled(v1.z, v1.w, kScaleW, p1[3], p2[3]);
      const int kb = c >> 3, cc = c & 7;
      uint8_t* img = sm + im * kLayerBytes + kb * kImgBytes + (nloc >> 3) * 1024 + (nloc & 7) * 128 + ((cc ^ (nloc & 7)) << 4);
      *reinterpret_cast<uint4*>(img) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
      *reinterpret_cast<uint4*>(img + 2 * kImgBytes) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
    }
  }
  // SYN: the narrow layer's weights live where the (unused) loader ring would be, all x kScaleA (the loader emits the
  // scaled operand; ReLU commutes with the scaling).  Per pair of output columns (2k, 2k + 1) 20 floats: the 8 weights
  // (zero-padded) interleaved column by column, then the two biases and two zeros - operand pairs of packed FMAs.
  float* s_syn = reinterpret_cast<float*>(sm + kOffLd2);
  if (SYN) {
    for (int i = threadIdx.x; i < kD * 10; i += kThreads) {
      const int k = i / 20, r = i - k * 20, col = 2 * k + (r & 1), j = r >> 1;
      float v = 0.f;
      if (j < p.syn_k) v = __ldg(p.syn_W + (long long)col * p.ld_syn_W + j) * kScaleA;
      else if (j == 8) v = p.syn_b ? __ldg(p.syn_b + col) * kScaleA : 0.f;
      s_syn[i] = v;
    }
  }
  for (int i = threadIdx.x; i < kD; i += kThreads) {
    for (int l = 0; l < NL; ++l) s_const[l * kD + i] = p.bias[l] ? __ldg(p.bias[l] + i) * (l < NL - 1 ? kScaleA : 1.f) : 0.f;
    s_const[3 * kD + i] = TAIL == 1 ? __ldg(p.dot_w + i) : (p.gamma ? __ldg(p.gamma + i) : 1.f);
    s_const[4 * kD + i] = (TAIL == 0 && p.gamma) ? __ldg(p.beta + i) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long long pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const long long n_my = (p.num_tiles > pair) ? (p.num_tiles - pair + npairs - 1) / npairs : 0;   // tile j -> slot j & 1
  constexpr int kOps = K2 ? 2 : 1;                  // operands of the first layer

  if (warp < kLoaderWarps) {
    // ======================= loaders =======================
    reg_dec<kRegsLd>();
    const int q = warp;
    const uint32_t buf0 = base + kOffLd2 + (uint32_t)(warp * kLoadBufs) * kChunkBytes;
    const int rl = lane >> 3, cj = lane & 7;
    const long long total = n_my * 4 * kOps;
    // item order = the MMA thread's order: per group of two tiles [op0 X][op0 Y][op1 X][op1 Y] (4 chunks each), so
    // that the second operand of a tile is converted while the other tile's first operand is being multiplied
    const long long full_groups = n_my >> 1;
    auto decode = [&](long long it, long long& j, int& op, int& c) {
      const long long per = 8 * kOps;
      if (it < full_groups * per) {
        const long long g = it / per;
        const int r = (int)(it - g * per);
        op = r >> 3; c = r & 3;
        j = 2 * g + ((r >> 2) & 1);
      } else {
        const int r = (int)(it - full_groups * per);
        op = r >> 2; c = r & 3;
        j = 2 * full_groups;
      }
    };
    const uint32_t a0_remote = map_to_leader(a0_full(0, 0));
    const uint64_t pol_keep = l2_policy_evict_last();
    // AGG: the two edge ids of this lane's row (thread = row; -1: none) for the tiles j with (j & 3) = 0 .. 3 - the two
    // tiles of the group being read back and the two of the next group, whose copies are issued up to three items ahead
    int ea0 = -1, ea1 = -1, ea2 = -1, ea3 = -1, eb0 = -1, eb1 = -1, eb2 = -1, eb3 = -1;
    // Both index levels are loaded a group before they are used and straight into the registers that will hold them, so
    // the loader never waits for them: at the end of group g the row pointers read at the end of group g - 1 address the
    // edge ids of group g + 2, and the row pointers of group g + 3 are requested.
    int rx0 = 0, rx1 = 0, ry0 = 0, ry1 = 0;           // row pointers (begin, end) of this lane's row in the two tiles of a group
    auto tile_row = [&](long long j) { return (pair + j * npairs) * kTileM + rank * 128 + q * 32 + lane; };
    auto load_rowptrs = [&](long long jx) {           // tiles jx, jx + 1
      rx0 = rx1 = ry0 = ry1 = 0;
      if (!AGG || PAIR) return;
      if (jx < n_my) { const long long row = tile_row(jx); if (row < p.M) { rx0 = __ldg(p.agg_rowptr + row); rx1 = __ldg(p.agg_rowptr + row + 1); } }
      if (jx + 1 < n_my) { const long long row = tile_row(jx + 1); if (row < p.M) { ry0 = __ldg(p.agg_rowptr + row); ry1 = __ldg(p.agg_rowptr + row + 1); } }
    };
    auto load_eids = [&](long long jx) {              // tiles jx (even), jx + 1 from rx / ry
      if (!AGG || PAIR) return;
      if (jx & 2) {
        ea2 = eb2 = ea3 = eb3 = -1;
        if (rx1 > rx0) ea2 = __ldg(p.agg_eid + rx0);
        if (rx1 > rx0 + 1) eb2 = __ldg(p.agg_eid + rx0 + 1);
        if (ry1 > ry0) ea3 = __ldg(p.agg_eid + ry0);
        if (ry1 > ry0 + 1) eb3 = __ldg(p.agg_eid + ry0 + 1);
      } else {
        ea0 = eb0 = ea1 = eb1 = -1;
        if (rx1 > rx0) ea0 = __ldg(p.agg_eid + rx0);
        if (rx1 > rx0 + 1) eb0 = __ldg(p.agg_eid + rx0 + 1);
        if (ry1 > ry0) ea1 = __ldg(p.agg_eid + ry0);
        if (ry1 > ry0 + 1) eb1 = __ldg(p.agg_eid + ry0 + 1);
      }
    };
    auto ids_a = [&](long long j) { const int k = (int)(j & 3); return k == 0 ? ea0 : k == 1 ? ea1 : k == 2 ? ea2 : ea3; };
    auto ids_b = [&](long long j) { const int k = (int)(j & 3); return k == 0 ? eb0 : k == 1 ? eb1 : k == 2 ? eb2 : eb3; };
    if (AGG) { load_rowptrs(0); load_eids(0); load_rowptrs(2); load_eids(2); load_rowptrs(4); }
    float x2[AGG ? 32 : 1];                           // AGG: the row's second edge row, columns 32 c .. 32 c + 31 of the item
    auto load_x2 = [&](long long it) {                // requested an item ahead: the wait for the slot hides the latency
      if (!AGG || it >= total) return;
      long long j; int op, c;
      decode(it, j, op, c);
      if (op != 0) return;
      const float* s2 = nullptr;
      if (PAIR) {
        const long long row = tile_row(j);
        if (row < p.M) s2 = p.A + (2 * row + 1) * p.lda + c * 32;
      } else {
        const int e = ids_b(j);
        if (e >= 0) s2 = p.A + (long long)e * p.lda + c * 32;
      }
      if (s2) {
#pragma unroll
        for (int t = 0; t < 4; ++t) ldg256_stream(s2 + 8 * t, x2 + 8 * t);
      } else {
#pragma unroll
        for (int t = 0; t < 32; ++t) x2[t] = 0.f;
      }
    };
    auto issue = [&](long long it, int b) {
      if (it < total) {
        long long j; int op, c;
        decode(it, j, op, c);
        const long long tile = pair + j * npairs;
        const long long row0 = tile * kTileM + rank * 128 + q * 32;
        const float* src = op ? p.A2 : p.A;
        const long long ld = op ? p.lda2 : p.lda;
        const uint32_t dst0 = buf0 + (uint32_t)b * kChunkBytes;
        if (PAIR && op == 0) {                        // row m's first edge row: slot 2m
          const float* s0 = src + 2 * row0 * ld + c * 32 + cj * 4;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = i * 4 + rl;
            const bool in = row0 + r < p.M;
            cp_async16(dst0 + (uint32_t)(r * 128 + ((cj ^ (r & 7)) << 4)), in ? s0 + 2 * r * ld : src, in ? 16u : 0u);
          }
        } else if (AGG && op == 0) {
          const int mine = ids_a(j);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = i * 4 + rl;
            const int e = __shfl_sync(0xffffffffu, mine, r);
            cp_async16(dst0 + (uint32_t)(r * 128 + ((cj ^ (r & 7)) << 4)), src + (long long)(e < 0 ? 0 : e) * ld + c * 32 + cj * 4, e < 0 ? 0u : 16u);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = i * 4 + rl;
            const long long row = row0 + r;
            const long long rc = row < p.M ? row : p.M - 1;
            cp_async16_hint(dst0 + (uint32_t)(r * 128 + ((cj ^ (r & 7)) << 4)), src + rc * ld + c * 32 + cj * 4, row < p.M ? 16u : 0u, pol_keep);
          }
        }
      }
      cp_async_commit();
    };
    if (!SYN) {
#pragma unroll
      for (int b = 0; b < kLoadBufs; ++b) issue(b, b);
    }
    int b = 0;
    float xin[8];                                     // SYN: this lane's input row (thread = row)
    load_x2(0);
    for (long long it = 0; it < total; ++it) {
      long long j; int op, c;
      decode(it, j, op, c);
      if (!SYN) asm volatile("cp.async.wait_group %0;" ::"n"(kLoadBufs - 1) : "memory");
      __syncwarp();
      const int S = (int)(j & 1);
      if (SYN && c == 0) {
        const long long row = (pair + j * npairs) * kTileM + rank * 128 + q * 32 + lane;
#pragma unroll
        for (int t = 0; t < 8; ++t) xin[t] = (row < p.M && t < p.syn_k) ? __ldg(p.A + row * p.lda + t) : 0.f;
      }
      const uint32_t u = (uint32_t)(j >> 1);          // tiles this slot has seen
      if (op == 0) mbar_wait(a_empty(S, c), (u & 1u) ^ 1u);   // the slot's previous tile has read chunk c
      else mbar_wait(a_mid(S, c), u & 1u);                    // this tile's first-operand MMAs have read chunk c
      tc_fence_after();
      const uint8_t* buf = sm + kOffLd2 + (warp * kLoadBufs + b) * kChunkBytes + lane * 128;
      const uint32_t ta = tmem_base + (uint32_t)S * 256 + 128 + ((uint32_t)(q * 32) << 16) + (uint32_t)c * 16;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t p1[8], p2[8];
        if (SYN) {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {           // columns c * 32 + half * 16 + 2 jj, + 1 (one packed lane each)
            const float* w = s_syn + (c * 16 + half * 8 + jj) * 20;
            float2 acc = *reinterpret_cast<const float2*>(w + 16);
#pragma unroll
            for (int t = 0; t < 8; t += 2) {
              const float4 wt = *reinterpret_cast<const float4*>(w + 2 * t);     // weights t, t + 1 of both columns
              acc = __ffma2_rn(dup2(xin[t]), make_float2(wt.x, wt.y), acc);
              acc = __ffma2_rn(dup2(xin[t + 1]), make_float2(wt.z, wt.w), acc);
            }
            split2(relu_nan(acc.x), relu_nan(acc.y), p1[jj], p2[jj]);
          }
        } else {
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float4 x = *reinterpret_cast<const float4*>(buf + (((half * 4 + jj) ^ (lane & 7)) << 4));
            float2 xa = make_float2(x.x, x.y), xb = make_float2(x.z, x.w);
            if (PAIR && op == 0) {                    // (0 + a) + b, a = row 2m (horizontal), b = row 2m + 1 (vertical)
              const float* y = x2 + 16 * half + 4 * jj;
              xa = __fadd2_rn(__fadd2_rn(dup2(0.f), xa), pair2(y));
              xb = __fadd2_rn(__fadd2_rn(dup2(0.f), xb), pair2(y + 2));
            } else if (AGG && op == 0) {              // (0 + a) + b: the ordered sum of the row's edges
              const float* y = x2 + 16 * half + 4 * jj;
              xa = __fadd2_rn(xa, pair2(y));
              xb = __fadd2_rn(xb, pair2(y + 2));
            }
            split2(__fmul2_rn(xa, dup2(kScaleA)), p1[2 * jj], p2[2 * jj]);
            split2(__fmul2_rn(xb, dup2(kScaleA)), p1[2 * jj + 1], p2[2 * jj + 1]);
          }
        }
        tmem_st8(ta + half * 8, p1);
        tmem_st8(ta + 64 + half * 8, p2);
      }
      // AGG: the last item of a group has been read back - its tiles' ids are dead, those of the group after the next
      // take their place (the copies of the next group's first items are already in flight with ids loaded a group ago)
      if (AGG && !PAIR && op == kOps - 1 && c == 3 && (((j & 1) == 1) || j + 1 >= n_my)) {
        const long long jx = (j | 1) + 3;             // first tile of group g + 2 (g = this group)
        load_eids(jx);
        load_rowptrs(jx + 2);
      }
      load_x2(it + 1);                                // x2 of this item is consumed: the next item's second source
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive_remote(a0_remote + 144u * (uint32_t)S + 8u * (uint32_t)c);
      __syncwarp();
      if (!SYN) issue(it + kLoadBufs, b);
      b = (b + 1 == kLoadBufs) ? 0 : b + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp < kEpiWarp0) {
    // ======================= MMA issuer =======================
    reg_dec<kRegsMma>();
    if (rank == 0 && warp == kMmaWarp && lane == 0) {
      const uint64_t desc0 = make_desc(base);
      const long long groups = (n_my + 1) >> 1;
      auto mma_chunk = [&](uint32_t d_tmem, uint32_t a_base, uint64_t desc_img, int c, bool first_of_layer) {
#pragma unroll
        for (int k2 = 0; k2 < 2; ++k2) {
          const int ks = 2 * c + k2;
          const uint32_t a1 = a_base + (uint32_t)ks * 8, a2 = a1 + 64;
          const uint64_t w1 = desc_img + (uint64_t)(((ks >> 2) * kImgBytes + (ks & 3) * 32) >> 4);
          const uint64_t w2 = w1 + (uint64_t)((2 * kImgBytes) >> 4);
          umma_f16_pair(d_tmem, a1, w2, kInstrDesc, !(first_of_layer && ks == 0));
          umma_f16_pair(d_tmem, a2, w1, kInstrDesc, 1);
          umma_f16_pair(d_tmem, a1, w1, kInstrDesc, 1);
        }
      };
#pragma unroll 1
      for (long long g = 0; g < groups; ++g) {
        // phases of a group: (layer 0, operand 0) [(layer 0, operand 1)] layer 1 ... - each over both slots
#pragma unroll 1
        for (int ph = 0; ph < NL + kOps - 1; ++ph) {
          const int l = ph < kOps ? 0 : ph - kOps + 1;
          const int op = ph < kOps ? ph : 0;
#pragma unroll 1
          for (int S = 0; S < 2; ++S) {
            if (2 * g + S >= n_my) continue;
            const uint32_t d_tmem = tmem_base + (uint32_t)S * 256;
            const uint32_t a_base = d_tmem + 128;
            if (l == 0) {
              if (op == 0 && g > 0) {               // the slot's previous tile has copied its last accumulator out
                mbar_wait(d_free(S), (uint32_t)((g - 1) & 1));
                tc_fence_after();
              }
              const uint64_t desc_img = desc0 + (uint64_t)((op * kLayerBytes) >> 4);
#pragma unroll 1
              for (int c = 0; c < 4; ++c) {
                mbar_wait(a0_full(S, c), (uint32_t)((g * kOps + op) & 1));
                tc_fence_after();
                mma_chunk(d_tmem, a_base, desc_img, c, op == 0);
                if (K2 && op == 0) umma_commit_pair(a_mid(S, c));        // the second operand may overwrite chunk c
              }
              if (op == kOps - 1) umma_commit_pair(d_full(S));
            } else {
              const uint64_t desc_img = desc0 + (uint64_t)(((l + (K2 ? 1 : 0)) * kLayerBytes) >> 4);
#pragma unroll 1
              for (int c = 0; c < 4; ++c) {
                mbar_wait(ae_full(S, c), (uint32_t)((g * (NL - 1) + (l - 1)) & 1));
                tc_fence_after();
                mma_chunk(d_tmem, a_base, desc_img, c, true);
                if (l == NL - 1) umma_commit_pair(a_empty(S, c));
              }
              umma_commit_pair(d_full(S));
            }
          }
        }
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    reg_inc<kRegsEp>();
    const int ew = warp - kEpiWarp0;
    const int q = warp & 3, hf = ew >> 2;
    uint8_t* slots = sm + kOffEp2 + ew * 2 * kSlotBytes;
    const uint32_t slots_u = base + kOffEp2 + (uint32_t)ew * 2 * kSlotBytes;
    float* xchg = reinterpret_cast<float*>(sm + kOffXchg2);
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int rl = lane >> 2, cc = lane & 3;
    const uint32_t ae_remote = map_to_leader(ae_full(0, 0)), dfree_remote = map_to_leader(d_free(0));
    auto slot_off = [](int r, int ch) { return (uint32_t)(r * 64 + ((ch ^ ((r >> 1) & 3)) << 4)); };
    auto read_slot = [&](const uint8_t* slot, float* v) {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const float4 x = *reinterpret_cast<const float4*>(slot + slot_off(lane, ch));
        v[4 * ch] = x.x; v[4 * ch + 1] = x.y; v[4 * ch + 2] = x.z; v[4 * ch + 3] = x.w;
      }
    };
    auto tile_row0 = [&](long long j) { return (pair + j * npairs) * kTileM + rank * 128 + q * 32; };
    uint32_t soff[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) soff[i] = slot_off(rl + 8 * i, cc);
    const int lane_col = 16 * hf + 4 * cc;
    const uint64_t pol_drop = l2_policy_evict_first();

    // residual stream: step k (= 4 j + c over the pair's tiles) uses slot k & 1, two steps in flight, FIFO
    long long res_issued = 0, res_consumed = 0;
    const long long res_total = RES ? 4 * n_my : 0;
    auto issue_res = [&]() {
      if (res_issued < res_total) {
        const long long j = res_issued >> 2;
        const int c = (int)(res_issued & 3);
        const long long r0 = tile_row0(j);
        const uint32_t dst = slots_u + (uint32_t)(res_issued & 1) * kSlotBytes;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          long long g = r0 + rl + 8 * i;
          g = g < p.M ? g : p.M - 1;
          cp_async16_hint(dst + soff[i], p.residual + g * p.ld_res + lane_col + 32 * c, 16u, pol_drop);
        }
      }
      cp_async_commit();                            // always: uniform group counting
      ++res_issued;
    };
    auto emit_chunk = [&](const float* vc, const float* s_bias, int S, int c) {
      const int col0 = 32 * c + 16 * hf;
      uint32_t p1[8], p2[8];
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        const float4 b4 = *reinterpret_cast<const float4*>(s_bias + col0 + 4 * j4);
        const float2 ya = __ffma2_rn(pair2(vc + 4 * j4), dup2(1.f / kScaleW), make_float2(b4.x, b4.y));
        const float2 yb = __ffma2_rn(pair2(vc + 4 * j4 + 2), dup2(1.f / kScaleW), make_float2(b4.z, b4.w));
        split2(relu_nan(ya.x), relu_nan(ya.y), p1[2 * j4], p2[2 * j4]);
        split2(relu_nan(yb.x), relu_nan(yb.y), p1[2 * j4 + 1], p2[2 * j4 + 1]);
      }
      const uint32_t ta = lane_addr + (uint32_t)S * 256 + 128 + (uint32_t)(16 * c + 8 * hf);
      tmem_st8(ta, p1);
      tmem_st8(ta + 64, p2);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive_remote(ae_remote + 144u * (uint32_t)S + 8u * (uint32_t)c);
    };
    uint32_t dcnt0 = 0, dcnt1 = 0;
    auto wait_acc = [&](int S, float* v) {
      mbar_wait(d_full(S), (S ? dcnt1 : dcnt0) & 1u);
      if (S) ++dcnt1; else ++dcnt0;
      tc_fence_after();
      const uint32_t d_addr = lane_addr + (uint32_t)S * 256;
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld16(d_addr + 32 * c + 16 * hf, v + 16 * c);
      tmem_ld_wait();
    };

    const long long groups = (n_my + 1) >> 1;
    if (RES) { issue_res(); issue_res(); }
#pragma unroll 1
    for (long long g = 0; g < groups; ++g) {
      const bool hasY = 2 * g + 1 < n_my;
      // ---- hidden layers
#pragma unroll 1
      for (int l = 0; l < NL - 1; ++l) {
#pragma unroll 1
        for (int S = 0; S < 2; ++S) {
          if (S == 1 && !hasY) break;
          float v[64];
          wait_acc(S, v);
#pragma unroll
          for (int c = 0; c < 4; ++c) emit_chunk(v + 16 * c, s_const + l * kD, S, c);
        }
      }
      // ---- last layer
#pragma unroll 1
      for (int S = 0; S < 2; ++S) {
        if (S == 1 && !hasY) break;
        const long long row0 = tile_row0(2 * g + S);
        const bool tile_full = row0 + 32 <= p.M;
        float x[64];
        wait_acc(S, x);
        tc_fence_before();
        mbar_arrive_remote(dfree_remote + 144u * (uint32_t)S);
        const float* s_bias = s_const + (NL - 1) * kD;
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 32 * c + 16 * hf + 4 * j4);
            float* xx = x + 16 * c + 4 * j4;
            set2(xx, __ffma2_rn(pair2(xx), dup2(kUnscaleD), make_float2(b4.x, b4.y)));
            set2(xx + 2, __ffma2_rn(pair2(xx + 2), dup2(kUnscaleD), make_float2(b4.z, b4.w)));
          }
        float* xa = xchg + (ew * 32 + lane);
        float* xb = xchg + (kEpiWarps * 32) + (ew * 32 + lane);
        const int partner = (ew ^ 4) * 32 + lane;
        if (TAIL == 1) {
          float acc = 0.f;
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) acc = fmaf(relu_nan(x[16 * c + jj]), s_const[3 * kD + 32 * c + 16 * hf + jj], acc);
          const long long tcount = 2 * g + S;         // slot alternates per tile: one barrier per tile
          float* mine = (tcount & 1) ? xb : xa;
          *mine = acc;
          named_bar_sync(1 + q, 64);
          if (hf == 0) {
            const float other = xchg[((tcount & 1) ? kEpiWarps * 32 : 0) + partner];
            const long long gr = row0 + lane;
            if (gr < p.M) p.Y[gr * p.ldy] = acc + other + (p.dot_b ? __ldg(p.dot_b) : 0.f);
          }
          continue;
        }
        if (p.gamma) {
          const float mu = row_mean(x, xa, xchg + partner, q);
          const float rstd = row_rstd(x, mu, xb, xchg + kEpiWarps * 32 + partner, q, p.eps);
          normalise(x, rstd, s_const + 3 * kD + 16 * hf, s_const + 4 * kD + 16 * hf);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          // residual step k = 4 (2 g + S) + c lives in slot k & 1 = c & 1; without a residual the slot is only the
          // transpose tile of the output
          uint8_t* slot = slots + (c & 1) * kSlotBytes;
          if (RES) {
            asm volatile("cp.async.wait_group 1;" ::: "memory");      // the older of the two groups in flight
            ++res_consumed;
            __syncwarp();
            float rsd[16];
            read_slot(slot, rsd);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) set2(x + 16 * c + jj, __fadd2_rn(pair2(x + 16 * c + jj), pair2(rsd + jj)));
            __syncwarp();
          }
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
            *reinterpret_cast<float4*>(slot + slot_off(lane, ch)) =
                make_float4(x[16 * c + 4 * ch], x[16 * c + 4 * ch + 1], x[16 * c + 4 * ch + 2], x[16 * c + 4 * ch + 3]);
          __syncwarp();
          float4 o[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) o[i] = *reinterpret_cast<const float4*>(slot + soff[i]);
          float* yrow = p.Y + (row0 + rl) * p.ldy + 32 * c + lane_col;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (tile_full || row0 + rl + 8 * i < p.M) stg_hint(reinterpret_cast<float4*>(yrow + (long long)(8 * i) * p.ldy), o[i], pol_drop);
          __syncwarp();
          if (RES) issue_res();                        // the slot is free: next step of the stream
        }
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    (void)res_consumed;
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

template <int NL, bool K2, bool RES, int TAIL, bool SYN = false, bool AGG = false, bool PAIR = false>
static int launch_spec2n(const Params& p, cudaStream_t st) {
  // (the kernel's own layout: weight images, loader ring, 2 slots per epilogue warp, constants, barriers, slack)
  constexpr int kSmem2n = (NL + (K2 ? 1 : 0)) * kLayerBytes + kLoaderWarps * kLoadBufs * kChunkBytes + kEpiWarps * 2 * kSlotBytes +
                          5 * kD * 4 + 2 * kEpiWarps * 32 * 4 + 320 + 1024;
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(tc_chain2n_kernel<NL, K2, RES, TAIL, SYN, AGG, PAIR>, kSmem2n, "tc_chain2n")) return rc_attr;
  long long pairs = p.num_tiles < kNumSMs / 2 ? p.num_tiles : kNumSMs / 2;
  tc_chain2n_kernel<NL, K2, RES, TAIL, SYN, AGG, PAIR><<<(unsigned)(2 * pairs), kThreads, kSmem2n, st>>>(p);
  return check_launch("tc_chain2n_kernel");
}

template <int SPEC, bool STASH = false, bool PSUM = false>
static int launch_spec2(const Params& p, cudaStream_t st) {
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(tc_chain2_kernel<SPEC, STASH, PSUM>, kSmemBytes, "tc_chain2")) return rc_attr;
  long long pairs = p.num_tiles < kNumSMs / 2 ? p.num_tiles : kNumSMs / 2;
  tc_chain2_kernel<SPEC, STASH, PSUM><<<(unsigned)(2 * pairs), kThreads, kSmemBytes, st>>>(p);
  return check_launch("tc_chain2_kernel");
}

template <int SPEC>
static int launch_spec(const Params& p, cudaStream_t st) {
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(tc_chain_kernel<SPEC>, kSmemBytes, "tc_chain")) return rc_attr;
  long long pairs = p.num_tiles < kNumSMs / 2 ? p.num_tiles : kNumSMs / 2;
  tc_chain_kernel<SPEC><<<(unsigned)(2 * pairs), kThreads, kSmemBytes, st>>>(p);
  return check_launch("tc_chain_kernel");
}

// picks the specialised instantiation when the launch has exactly its shape (Spec<> above)
static int launch(const Params& p, cudaStream_t st) {
  if (p.st_a1) {                                  // training forward (form validated by the caller)
    return (p.g1 && p.i0) ? launch_spec2<1, true>(p, st) : launch_spec2<2, true>(p, st);
  }
  if (p.multi) return launch_spec<6>(p, st);
  if (p.edge_slots) {                             // only the two-tile kernel knows padding slots (form validated by the caller)
    if (!p.A) return p.edge_slots == 2 ? launch_spec2<7, false, true>(p, st) : launch_spec2<7>(p, st);
    return p.edge_slots == 2 ? launch_spec2<1, false, true>(p, st) : launch_spec2<1>(p, st);
  }
  if (!p.A) {
    static const bool two = []() { const char* e = getenv("GNC_CHAIN_TWO_TILES"); return !e || e[0] != '0'; }();
    return two ? launch_spec2<7>(p, st) : launch_spec<7>(p, st);
  }
  if (p.A2 && p.paired) return launch_spec2n<3, true, true, 0, false, true, true>(p, st);
  if (p.A2 && p.agg_rowptr) return launch_spec2n<3, true, true, 0, false, true>(p, st);
  if (p.A2) return launch_spec2n<3, true, true, 0>(p, st);
  if (p.syn_W) return launch_spec2n<2, false, false, 0, true>(p, st);     // (shape validated by the caller)
  if (p.trace && p.nlayers == 3 && p.g0 && p.i0 && p.g1 && p.i1 && p.residual && !p.res_idx && p.gamma && !p.dot_w)
    return launch_spec<8>(p, st);
  if (!p.trace) {
    const bool ln = p.gamma != nullptr, dot = p.dot_w != nullptr, res = p.residual != nullptr;
    static const bool two_tiles = []() { const char* e = getenv("GNC_CHAIN_TWO_TILES"); return !e || e[0] != '0'; }();
    if (p.nlayers == 3 && p.g0 && p.i0 && p.g1 && p.i1 && res && !p.res_idx && ln && !dot)
      return two_tiles ? launch_spec2<1>(p, st) : launch_spec<1>(p, st);
    if (p.nlayers == 3 && p.g0 && !p.i0 && !p.g1 && res && !p.res_idx && ln && !dot)
      return two_tiles ? launch_spec2<2>(p, st) : launch_spec<2>(p, st);
    if (p.A2) return launch_spec2n<3, true, true, 0>(p, st);     // (shape validated by the caller)
    if (two_tiles && p.nlayers == 2 && !p.g0 && !p.g1 && res && !p.res_idx && ln && !dot) return launch_spec2n<2, false, true, 0>(p, st);
    if (two_tiles && p.nlayers == 2 && !p.g0 && !p.g1 && !res && ln && !dot) return launch_spec2n<2, false, false, 0>(p, st);
    if (two_tiles && p.nlayers == 2 && !p.g0 && !p.g1 && !res && !ln && dot) return launch_spec2n<2, false, false, 1>(p, st);
    if (p.nlayers == 2 && !p.g0 && !p.g1 && res && ln && !dot) return launch_spec<3>(p, st);
    if (p.nlayers == 2 && !p.g0 && !p.g1 && !res && ln && !dot) return launch_spec<4>(p, st);
    if (p.nlayers == 2 && !p.g0 && !p.g1 && !res && !ln && dot) return launch_spec<5>(p, st);
  }
  return launch_spec<0>(p, st);
}

}  // namespace chain
}  // namespace gnc

using namespace gnc;

extern "C" int gnc_tc_mlp_chain_f32(const float* A, int64_t lda, int64_t M, const gnc_tc_chain_t* ch, float* Y, int64_t ldy,
                                    gnc_stream_t stream) {
  GNC_REQUIRE(ch && M >= 0, "tc_mlp_chain: bad arguments");
  GNC_REQUIRE(ch->nlayers >= 2 && ch->nlayers <= chain::kMaxLayers, "tc_mlp_chain: 2 or 3 layers");
  if (M == 0) return GNC_OK;                          // (empty tensors have no pointers: an edge-less graph)
  GNC_REQUIRE(Y, "tc_mlp_chain: null output");
  chain::Params p = {};
  p.A = A; p.lda = lda; p.M = M; p.nlayers = ch->nlayers;
  auto ok4 = [](const float* q, int64_t ld) { return !q || (aligned16(q) && ld % 4 == 0 && ld >= chain::kD); };
  if (A && ch->narrow_W) {
    /* validated with the narrow-first-layer fields below */
  } else if (A) {
    GNC_REQUIRE(lda >= chain::kD && lda % 4 == 0 && aligned16(A), "tc_mlp_chain: A rows must be 16-byte aligned");
    GNC_REQUIRE(!ch->gather2, "tc_mlp_chain: gather2 belongs to the pre-stage form (A == NULL)");
  } else {
    // pre-stage form: the first operand is relu(gather2[idx2] + gather0[idx0] + gather1[idx1] + pre_bias)
    GNC_REQUIRE(ch->nlayers == 2 && ch->gather0 && ch->gather0_idx && ch->gather1 && ch->gather1_idx && ch->gather2 &&
                ch->gather2_idx && ch->gamma && ch->residual && ch->residual_idx && !ch->dot_w,
                "tc_mlp_chain: the pre-stage form takes three indexed gathers, two layers, LayerNorm and an indexed residual");
    GNC_REQUIRE(ok4(ch->gather2, ch->ld_gather2), "tc_mlp_chain: gather2 rows must be 16-byte aligned, 128 wide");
    p.g2 = ch->gather2; p.i2 = ch->gather2_idx; p.ld_g2 = ch->ld_gather2; p.pre_bias = ch->pre_bias;
  }
  for (int l = 0; l < ch->nlayers; ++l) {
    GNC_REQUIRE(ch->W[l] && aligned16(ch->W[l]) && ch->ldw[l] >= chain::kD && ch->ldw[l] % 4 == 0, "tc_mlp_chain: bad weight pointer / stride");
    p.W[l] = ch->W[l]; p.ldw[l] = ch->ldw[l]; p.bias[l] = ch->bias[l];
  }
  if (ch->narrow_W) {
    // narrow first layer folded into the launch: relu(A[:, :k] narrow_W^T + narrow_b) -> 2 layers -> LayerNorm (encoders)
    GNC_REQUIRE(A && ch->narrow_k >= 1 && ch->narrow_k <= 8 && lda >= ch->narrow_k && ch->ld_narrow_W >= ch->narrow_k,
                "tc_mlp_chain: narrow first layer takes 1..8 input columns");
    GNC_REQUIRE(ch->nlayers == 2 && !ch->gather0 && !ch->gather1 && !ch->operand2 && ch->gamma && !ch->residual && !ch->dot_w,
                "tc_mlp_chain: the narrow-first-layer form is narrow layer + 2 layers + LayerNorm");
    p.syn_W = ch->narrow_W; p.ld_syn_W = ch->ld_narrow_W; p.syn_b = ch->narrow_b; p.syn_k = ch->narrow_k;
  }
  if (ch->operand2) {
    // two-operand first layer (the node processor's cat([x, agg]) @ V0^T): three layers, LayerNorm, residual by row
    GNC_REQUIRE(A && ch->nlayers == 3 && !ch->gather0 && !ch->gather1 && ch->gamma && ch->residual && !ch->residual_idx && !ch->dot_w,
                "tc_mlp_chain: operand2 takes the form 3 layers + LayerNorm + residual by row, without gathered addends");
    GNC_REQUIRE(ok4(ch->operand2, ch->ld_operand2) && ch->W_operand2 && aligned16(ch->W_operand2) && ch->ldw_operand2 >= chain::kD &&
                ch->ldw_operand2 % 4 == 0, "tc_mlp_chain: operand2 / W_operand2 must be 16-byte aligned, 128 wide");
    p.A2 = ch->operand2; p.lda2 = ch->ld_operand2; p.W_A2 = ch->W_operand2; p.ldw_A2 = ch->ldw_operand2;
    if (ch->agg_rowptr) {
      GNC_REQUIRE(ch->agg_eid && lda % 8 == 0 && ((uintptr_t)A) % 32 == 0,
                  "tc_mlp_chain: the aggregated operand needs agg_eid and 32-byte aligned edge rows (pitch a multiple of 8)");
      p.agg_rowptr = ch->agg_rowptr; p.agg_eid = ch->agg_eid;
    }
    if (ch->paired_operand) {
      GNC_REQUIRE(!ch->agg_rowptr && lda % 8 == 0 && ((uintptr_t)A) % 32 == 0,
                  "tc_mlp_chain: the paired operand excludes agg_rowptr and needs 32-byte aligned slot rows (pitch a multiple of 8)");
      p.paired = 1;
    }
  } else {
    GNC_REQUIRE(!ch->agg_rowptr && !ch->paired_operand, "tc_mlp_chain: agg_rowptr / paired_operand belong to the two-operand form");
  }
  if (ch->edge_slots) {
    // paired destination slots: the edge processor's two forms (three layers with gathers P[src], Q[dst], residual by row;
    // or the pre-stage form of block 0)
    GNC_REQUIRE(ch->edge_slots == 1 || ch->edge_slots == 2, "tc_mlp_chain: edge_slots is 0, 1 or 2");
    GNC_REQUIRE(ch->gather0 && ch->gather0_idx && ch->gather1 && ch->gather1_idx && ch->gamma && ch->residual && !ch->dot_w &&
                !ch->operand2 && !ch->narrow_W && !ch->stash_a1 &&
                ((A && ch->nlayers == 3 && !ch->residual_idx) || (!A && ch->nlayers == 2)),
                "tc_mlp_chain: edge_slots takes the edge processor's forms (two indexed gathers, LayerNorm, residual)");
    GNC_REQUIRE(ch->edge_slots == 1 || M % 2 == 0, "tc_mlp_chain: pair sums need an even number of slot rows");
    p.edge_slots = ch->edge_slots;
  }
  GNC_REQUIRE(ok4(ch->gather0, ch->ld_gather0) && ok4(ch->gather1, ch->ld_gather1) && ok4(ch->residual, ch->ld_residual),
              "tc_mlp_chain: addend / residual rows must be 16-byte aligned, 128 wide");
  p.g0 = ch->gather0; p.i0 = ch->gather0_idx; p.ld_g0 = ch->ld_gather0;
  p.g1 = ch->gather1; p.i1 = ch->gather1_idx; p.ld_g1 = ch->ld_gather1;
  p.gamma = ch->gamma; p.beta = ch->beta; p.eps = ch->eps;
  p.residual = ch->residual; p.res_idx = ch->residual_idx; p.ld_res = ch->ld_residual;
  p.dot_w = ch->dot_w; p.dot_b = ch->dot_b;
  GNC_REQUIRE(!p.gamma || p.beta, "tc_mlp_chain: LayerNorm needs gamma and beta");
  if (p.dot_w) {
    GNC_REQUIRE(!p.gamma && !p.residual && ldy >= 1, "tc_mlp_chain: the dot tail excludes LayerNorm / residual");
  } else {
    GNC_REQUIRE(ldy >= chain::kD && ldy % 4 == 0 && aligned16(Y), "tc_mlp_chain: Y rows must be 16-byte aligned");
  }
  p.Y = Y; p.ldy = ldy;
  p.num_tiles = (M + chain::kTileM - 1) / chain::kTileM;
  p.trace = chain::g_trace; p.trace_cap = chain::g_trace_cap;
  if (ch->stash_a1) {
    const bool edge_form = ch->gather0 && ch->gather0_idx && ch->gather1 && ch->gather1_idx;
    const bool node_form = ch->gather0 && !ch->gather0_idx && !ch->gather1;
    GNC_REQUIRE(A && ch->nlayers == 3 && (edge_form || node_form) && ch->gamma && ch->residual && !ch->residual_idx && !ch->dot_w &&
                !ch->operand2 && !ch->narrow_W,
                "tc_mlp_chain: the stash goes with 3 layers + addends (two indexed gathers, or one plain addend) + LayerNorm + "
                "residual by row");
    GNC_REQUIRE(ch->stash_a2 && ch->stash_z && ch->stash_mean && ch->stash_rstd && ch->ld_stash >= chain::kD && ch->ld_stash % 4 == 0 &&
                ch->ld_stash % 8 == 0 && ((uintptr_t)ch->stash_a1 | (uintptr_t)ch->stash_a2 | (uintptr_t)ch->stash_z) % 32 == 0,
                "tc_mlp_chain: stash_a1 / a2 / z must be 32-byte aligned [M, 128] row sets (pitch a multiple of 8), with mean and rstd [M]");
    p.st_a1 = ch->stash_a1; p.st_a2 = ch->stash_a2; p.st_z = ch->stash_z; p.ld_st = ch->ld_stash;
    p.st_mean = ch->stash_mean; p.st_rstd = ch->stash_rstd;
    p.trace = nullptr;
  }
  return chain::launch(p, (cudaStream_t)stream);
}

// Debug: CTA 0 of subsequent gnc_tc_mlp_chain_f32 launches records (clock64 << 8 | tag) events for
// chain::kTraceRoles roles into buf[role * cap + i] (device memory, zeroed by the caller).  NULL disables.
extern "C" int gnc_debug_chain_trace(unsigned long long* buf, int cap) {
  chain::g_trace = buf; chain::g_trace_cap = cap;
  return GNC_OK;
}

// Y_l[M, 128] = A[M, 128] * W_l[128, 128]^T (+ bias_l) for nsets = 2 or 3 weight sets in ONE launch of the
// chained kernel in multi mode: A is read from memory once and stays in tensor memory for all products.
extern "C" int gnc_tc_multi_chain_f32(const float* A, int64_t lda, int64_t M, int nsets, const float* const* W,
                                      const int64_t* ldw, const float* const* bias, float* const* Y, int64_t ldy,
                                      gnc_stream_t stream) {
  GNC_REQUIRE(nsets >= 2 && nsets <= chain::kMaxLayers && A && W && ldw && Y && M >= 0 && lda >= chain::kD && ldy >= chain::kD,
              "tc_multi_chain: need 2 or 3 weight sets");
  if (M == 0) return GNC_OK;
  GNC_REQUIRE(lda % 4 == 0 && aligned16(A) && ldy % 4 == 0, "tc_multi_chain: rows must be 16-byte aligned");
  chain::Params p = {};
  p.A = A; p.lda = lda; p.M = M; p.nlayers = nsets; p.multi = 1; p.ldy = ldy; p.eps = 1e-5f;
  for (int l = 0; l < nsets; ++l) {
    GNC_REQUIRE(W[l] && Y[l] && aligned16(W[l]) && aligned16(Y[l]) && ldw[l] % 4 == 0 && ldw[l] >= chain::kD,
                "tc_multi_chain: bad weight / output pointer");
    p.W[l] = W[l]; p.ldw[l] = ldw[l]; p.bias[l] = bias ? bias[l] : nullptr; p.Ym[l] = Y[l];
  }
  p.Y = Y[0];
  p.num_tiles = (M + chain::kTileM - 1) / chain::kTileM;
  return chain::launch(p, (cudaStream_t)stream);
}
