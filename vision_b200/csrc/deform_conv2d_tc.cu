// deform_conv2d_tc.cu — tcgen05 (5th-gen tensor core) path for deform_conv2d, 16-bit storage types.
//
// Reference: csrc/ops/cuda/deform_conv2d_kernel.cu:136-209 (deformable_im2col writes a
// [C_in*kh*kw, pixels] buffer to HBM) + :1234-1239 (cuBLAS addmm) + transpose/copy/bias passes.
//
// Here the op is ONE implicit GEMM whose gathered operand never touches HBM:
//     D[pixel, cout] = sum_k A[pixel, k] * Wt[cout, k],   k = (channel slab, tap, channel in slab)
//   * M = 128 output pixels (TMEM lanes), N = BN output channels (TMEM fp32 columns), K step 64;
//   * A tiles are SYNTHESISED by 8 gather warps: per (pixel, tap) the 4 bilinear corner offsets and
//     weights (x modulation mask) come from a per-CTA table built once; channels are the fastest
//     axis of a channels-last staging copy of the input, so every corner read is a 128-bit vector
//     load of 8 consecutive channels; the fp32 blend is rounded to bf16/fp16 and stored into the
//     128B-swizzled K-major shared-memory tile the tensor core descriptor expects;
//   * B (weights) tiles are pre-packed once per call into the exact swizzled shared-memory image,
//     so a stage is filled by one 1-D bulk async copy (TMA engine) completing on an mbarrier;
//   * one elected thread issues tcgen05.mma (cta_group::1, kind::f16, fp32 accumulate in TMEM);
//     tcgen05.commit hands stages back to the producers and signals the epilogue;
//   * epilogue: tcgen05.ld 32 lanes x 16 columns, + bias, round, coalesced NCHW stores.
// Pipeline: 3 stages x (A 16 KB + B BN*128 B), full(A)/full(B)/empty mbarriers per stage.
#include "async_copy.cuh"
#include <type_traits>

#include "common.cuh"
#include "dcn_params.h"

namespace vb200 {


namespace {

constexpr int TC_BM = 128, TC_GATHER_WARPS = 8;
constexpr int TC_GATHER_THREADS = TC_GATHER_WARPS * 32;
constexpr int TC_THREADS = TC_GATHER_THREADS + 64;          // + bulk-copy warp + MMA warp (CTA-pair kernel)
constexpr int TC1_GATHER_WARPS = 16;                         // single-CTA kernel: two groups of 8 gather warps
constexpr int TC1_GATHER_THREADS = TC1_GATHER_WARPS * 32;
constexpr int TC1_THREADS = TC1_GATHER_THREADS + 64;
// KB = K elements per pipeline stage: 64 (128-byte rows, SWIZZLE_128B) or 32 (64-byte rows, SWIZZLE_64B).
// The gather always works on 64-channel slabs (whole 128-byte lines); with KB = 32 one gather step
// fills two consecutive stages.  16-byte chunk c of row r is stored at chunk c ^ swz(r).
template <int KB> __host__ __device__ constexpr int tc_swz(int r) { return KB == 64 ? (r & 7) : ((r >> 1) & 3); }

// ---- pre-pass 1: NCHW -> NHWC (16-bit elements) -------------------------------------------
// 64 channels x 64 pixels per CTA; 32-bit global accesses on both sides (2 pixels in, 2 channels out),
// 128-byte rows per warp access.  Requires C % 64 == 0 and HW % 2 == 0 (else the scalar kernel below).
template <typename T>
__global__ void __launch_bounds__(256)
nchw_to_nhwc64_kernel(const T* __restrict__ in, T* __restrict__ out, int C, int HW) {
  __shared__ __align__(4) unsigned short tile[64][66];
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned short* __restrict__ src = reinterpret_cast<const unsigned short*>(in) + (int64_t)b * C * HW;
  unsigned short* __restrict__ dst = reinterpret_cast<unsigned short*>(out) + (int64_t)b * C * HW;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = warp + i * 8, p = p0 + 2 * lane;
    uint32_t v = 0u;
    if (p < HW) v = __ldg(reinterpret_cast<const uint32_t*>(src + (int64_t)(c0 + c) * HW + p));
    *reinterpret_cast<uint32_t*>(&tile[c][2 * lane]) = v;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int pl = warp + i * 8, p = p0 + pl;
    if (p < HW) {
      const uint32_t v = (uint32_t)tile[2 * lane][pl] | ((uint32_t)tile[2 * lane + 1][pl] << 16);
      *reinterpret_cast<uint32_t*>(dst + (int64_t)p * C + c0 + 2 * lane) = v;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
nchw_to_nhwc_kernel(const T* __restrict__ in, T* __restrict__ out, int C, int HW) {
  __shared__ T tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
  const T* __restrict__ src = in + (int64_t)b * C * HW;
  T* __restrict__ dst = out + (int64_t)b * C * HW;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + i * 8, p = p0 + tx;
    if (c < C && p < HW) tile[ty + i * 8][tx] = src[(int64_t)c * HW + p];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int p = p0 + ty + i * 8, c = c0 + tx;
    if (c < C && p < HW) dst[(int64_t)p * C + c] = tile[tx][ty + i * 8];
  }
}

// ---- pre-pass 2: weights [Cout][Cin][KK] -> swizzled K-major tiles ---------------------------
// K order: (64-channel slab, tap, half) -> stage q = (cslab*KK + tap) * (64/KB) + half; tile (nt, q) holds
// BN rows x KB k as the exact shared-memory image: byte = r*(2*KB) + ((kc/8) ^ swz(r))*16 + (kc%8)*2.
template <typename T, int KB>
__global__ void __launch_bounds__(256)
pack_weights_kernel(const T* __restrict__ w, T* __restrict__ packed, int Cout, int Cin, int KK, int BN) {
  const int64_t total = (int64_t)Cout * Cin * KK;
  constexpr int SPLIT = 64 / KB;
  const int n_q = (Cin / 64) * KK * SPLIT;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int tap = (int)(e % KK);
    const int ci = (int)((e / KK) % Cin);
    const int co = (int)(e / KK / Cin);
    const int nt = co / BN, r = co % BN;
    const int cslab = ci / 64, kc64 = ci % 64;
    const int half = kc64 / KB, kc = kc64 % KB;
    const int q = (cslab * KK + tap) * SPLIT + half;
    const int64_t tile_base = ((int64_t)nt * n_q + q) * BN * KB;
    const int off_bytes = r * (2 * KB) + (((kc >> 3) ^ tc_swz<KB>(r)) << 4) + ((kc & 7) << 1);
    packed[tile_base + (off_bytes >> 1)] = w[e];
  }
}

// ---- tcgen05 wrappers -------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_c), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// K-major swizzled shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm_100):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major: 1) | SBO>>4 [32,46) = bytes between 8-row
// groups (8 * row bytes) | version=1 [46,48) | layout_type [61,64): 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
template <int KB>
__device__ __forceinline__ uint64_t smem_desc_k(uint32_t smem_addr) {
  constexpr uint64_t sbo = (uint64_t)(8 * 2 * KB) >> 4;
  constexpr uint64_t layout = KB == 64 ? 2ull : 4ull;
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}

template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
  static constexpr uint32_t kFmt = 1;
  // packed 16-bit blend (HFMA2.BF16): weight pair x value pair + accumulator pair, one rounding to bf16 per step
  static __device__ __forceinline__ uint32_t dup(float w) { __nv_bfloat162 v = __float2bfloat162_rn(w); return *reinterpret_cast<uint32_t*>(&v); }
  static __device__ __forceinline__ uint32_t mul2(uint32_t w, uint32_t a) {
    __nv_bfloat162 r = __hmul2(*reinterpret_cast<__nv_bfloat162*>(&w), *reinterpret_cast<__nv_bfloat162*>(&a)); return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ uint32_t fma2p(uint32_t w, uint32_t a, uint32_t c) {
    __nv_bfloat162 r = __hfma2(*reinterpret_cast<__nv_bfloat162*>(&w), *reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&c));
    return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ float2 up(uint32_t u) { return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u)); }
  static __device__ __forceinline__ uint32_t pk(float a, float b) { __nv_bfloat162 v = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
};
template <> struct Elem<__half> {
  static constexpr uint32_t kFmt = 0;
  static __device__ __forceinline__ uint32_t dup(float w) { __half2 v = __float2half2_rn(w); return *reinterpret_cast<uint32_t*>(&v); }
  static __device__ __forceinline__ uint32_t mul2(uint32_t w, uint32_t a) {
    __half2 r = __hmul2(*reinterpret_cast<__half2*>(&w), *reinterpret_cast<__half2*>(&a)); return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ uint32_t fma2p(uint32_t w, uint32_t a, uint32_t c) {
    __half2 r = __hfma2(*reinterpret_cast<__half2*>(&w), *reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&c));
    return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ float2 up(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
  static __device__ __forceinline__ uint32_t pk(float a, float b) { __half2 v = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
};

struct __align__(16) TcEnt { int o[4]; float w[4]; };   // clamped corner pixel indices (y*W+x) + bilinear weights x mask

// BN = output channels per CTA: 128 / 256 (one accumulator, 3 stages) or 512 (two 256-column
// accumulators = all of TMEM, K depth 32, 4 stages (3 by override); the A tile is then gathered once per pixel tile).
template <typename T, int BN, int TC_STAGES, int KB>
__global__ void __launch_bounds__(TC1_THREADS, 1)
deform_conv2d_tc_kernel(const T* __restrict__ nhwc, const T* __restrict__ wpacked, const T* __restrict__ offset,
                        const T* __restrict__ mask, const T* __restrict__ bias, T* __restrict__ out, DcnParams p) {
  constexpr int ROW_BYTES = 2 * KB;
  constexpr int TC_A_BYTES = TC_BM * ROW_BYTES;
  constexpr int B_BYTES = BN * ROW_BYTES;
  constexpr int STAGE_BYTES = TC_A_BYTES + B_BYTES;
  constexpr int SPLIT = 64 / KB;                       // stages filled per 64-channel gather step
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* stages = smem;
  uint64_t* fullA = reinterpret_cast<uint64_t*>(stages + TC_STAGES * STAGE_BYTES);
  uint64_t* fullB = fullA + TC_STAGES;
  uint64_t* empty = fullB + TC_STAGES;
  uint64_t* accum_full = empty + TC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_full + 1);
  // [KK][128] sampling table, 32-byte aligned (entries are read as int4 + float4)
  TcEnt* tab = reinterpret_cast<TcEnt*>(stages + ((TC_STAGES * STAGE_BYTES + (3 * TC_STAGES + 1) * 8 + 16 + 31) & ~31));

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int KK = p.kh * p.kw;
  const int HWo = p.out_h * p.out_w, HWi = p.in_h * p.in_w;
  const int tiles_per_img = ceil_div(HWo, TC_BM);
  const int b = blockIdx.x / tiles_per_img;
  const int pix0 = (blockIdx.x % tiles_per_img) * TC_BM;
  const int nt = blockIdx.y;
  const int c_per_off = p.c_in / p.offset_groups;
  const int slabs_per_og = (c_per_off / 64) * KK;      // 64-channel gather steps per offset group
  const int n_q = (p.c_in / 64) * KK * SPLIT;          // pipeline stages consumed per tile

  if (tid == 0) {
    for (int s = 0; s < TC_STAGES; ++s) { mbar_init(&fullA[s], TC_GATHER_WARPS); mbar_init(&fullB[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(accum_full, 1);
    mbar_fence_init();
  }
  if (warp == TC1_GATHER_WARPS + 1) tmem_alloc(tmem_slot, BN);    // whole warp, .sync.aligned
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < TC1_GATHER_WARPS) {
    // ================= gather warps: build A tiles =================
    // Two groups of 8 warps take ALTERNATE 64-channel steps (group g owns the steps whose global index
    // is g mod 2): twice the warps in flight for the same instruction count — the kernel is bound by the
    // gather's issue rate (272 k warp instructions per tile at ~1.6 IPC), not by memory or the tensor pipe.
    const int group = warp >> 3, wg = warp & 7;
    // lane = (pixel sub-index pq, 16-byte chunk c): one warp load instruction reads four complete
    // 128-byte lines (4 pixels x 64 channels) instead of sixteen quarter lines.
    const int cchunk = lane & 7, pq = lane >> 3;
    const int prow0 = wg * 16 + pq;                          // + 4 * i, i = 0..3
    const T* __restrict__ in_b = nhwc + (int64_t)b * HWi * p.c_in;
    for (int og = 0; og < p.offset_groups; ++og) {
      // ---- sampling table for this offset group: [KK][128] ----
      asm volatile("bar.sync 1, %0;" ::"n"(TC1_GATHER_THREADS));     // previous table no longer read
      const T* __restrict__ off_b = offset + ((int64_t)b * p.offset_groups + og) * 2 * KK * HWo;
      const T* __restrict__ msk_b = p.use_mask ? mask + ((int64_t)b * p.offset_groups + og) * KK * HWo : nullptr;
      for (int e = tid; e < KK * TC_BM; e += TC1_GATHER_THREADS) {
        const int tap = e / TC_BM, px = e - tap * TC_BM;
        const int pix = pix0 + px;
        TcEnt se;
#pragma unroll
        for (int q = 0; q < 4; ++q) { se.o[q] = 0; se.w[q] = 0.f; }
        if (pix < HWo) {
          const int oy = pix / p.out_w, ox = pix - oy * p.out_w;
          const int i = tap / p.kw, j = tap - i * p.kw;
          const float oh = to_acc(off_b[(int64_t)(2 * tap) * HWo + pix]);
          const float ow = to_acc(off_b[(int64_t)(2 * tap + 1) * HWo + pix]);
          const float mv = p.use_mask ? to_acc(msk_b[(int64_t)tap * HWo + pix]) : 1.f;
          const float y = add_rn((float)(oy * p.stride_h - p.pad_h + i * p.dil_h), oh);
          const float x = add_rn((float)(ox * p.stride_w - p.pad_w + j * p.dil_w), ow);
          if (!(y <= -1.f || (float)p.in_h <= y || x <= -1.f || (float)p.in_w <= x)) {
            const int hl = (int)floorf(y), wl = (int)floorf(x);
            const int hh_i = hl + 1, wh_i = wl + 1;
            const float lh = y - (float)hl, lw = x - (float)wl;
            const float hh = 1.f - lh, hw = 1.f - lw;
            const bool t0 = hl >= 0, t1 = hh_i <= p.in_h - 1, l0 = wl >= 0, l1 = wh_i <= p.in_w - 1;
            const int hlc = max(hl, 0), hhc = min(hh_i, p.in_h - 1), wlc = max(wl, 0), whc = min(wh_i, p.in_w - 1);
            se.o[0] = (hlc * p.in_w + wlc) * p.c_in * 2; se.w[0] = (t0 && l0) ? mv * (hh * hw) : 0.f;
            se.o[1] = (hlc * p.in_w + whc) * p.c_in * 2; se.w[1] = (t0 && l1) ? mv * (hh * lw) : 0.f;
            se.o[2] = (hhc * p.in_w + wlc) * p.c_in * 2; se.w[2] = (t1 && l0) ? mv * (lh * hw) : 0.f;
            se.o[3] = (hhc * p.in_w + whc) * p.c_in * 2; se.w[3] = (t1 && l1) ? mv * (lh * lw) : 0.f;
          }
        }
        tab[e] = se;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(TC1_GATHER_THREADS));
      // ---- slabs of this offset group: channel slab outer, tap inner (L1 reuse across taps) ----
      const int slab_base = og * slabs_per_og;
      for (int sl = (slab_base + group) & 1; sl < slabs_per_og; sl += 2) {
        const int slab = slab_base + sl;
        const int cs_local = sl / KK, tap = sl - cs_local * KK;
        // corner offsets are 32-bit BYTE offsets (image < 2^30 elements): uniform 64-bit base + 32-bit offset
        const char* __restrict__ in_c = reinterpret_cast<const char*>(in_b + og * c_per_off + cs_local * 64);
        const uint32_t lane_off = (uint32_t)cchunk * 16u;
        uint4 v[4][4];                                       // [pixel][corner]
        float4 wq[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {                        // all 16 loads in flight before the blend
          const TcEnt* se = tab + tap * TC_BM + prow0 + 4 * i;
          const uint4 o = *reinterpret_cast<const uint4*>(se->o);
          wq[i] = *reinterpret_cast<const float4*>(se->w);
          v[i][0] = __ldg(reinterpret_cast<const uint4*>(in_c + (o.x + lane_off)));
          v[i][1] = __ldg(reinterpret_cast<const uint4*>(in_c + (o.y + lane_off)));
          v[i][2] = __ldg(reinterpret_cast<const uint4*>(in_c + (o.z + lane_off)));
          v[i][3] = __ldg(reinterpret_cast<const uint4*>(in_c + (o.w + lane_off)));
        }
        // this thread's 8 channels land in sub-stage (cchunk / (KB/8)) of the SPLIT stages of this step
        const int q0 = slab * SPLIT;
#pragma unroll
        for (int h = 0; h < SPLIT; ++h) {
          const int qq = q0 + h;
          mbar_wait(&empty[qq % TC_STAGES], ((uint32_t)(qq / TC_STAGES) & 1u) ^ 1u);
        }
        constexpr int CH_PER_ROW = KB / 8;                   // 16-byte chunks per tile row
        const int my_q = q0 + cchunk / CH_PER_ROW, my_chunk = cchunk % CH_PER_ROW;
        unsigned char* a_tile = stages + (my_q % TC_STAGES) * STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float wv[4] = {wq[i].x, wq[i].y, wq[i].z, wq[i].w};
          uint4 o;
          if (p.blend16) {
            // blend in the storage format (HFMA2): 16 instructions per 8 channels instead of 52 (unpack + FFMA2 + pack).  Every
            // step rounds to 16 bits - the A operand is rounded to that format anyway; the whole op stays inside its 1e-2 bound.
            const uint32_t w0 = Elem<T>::dup(wv[0]), w1 = Elem<T>::dup(wv[1]), w2_ = Elem<T>::dup(wv[2]), w3 = Elem<T>::dup(wv[3]);
            o.x = Elem<T>::fma2p(w3, v[i][3].x, Elem<T>::fma2p(w2_, v[i][2].x, Elem<T>::fma2p(w1, v[i][1].x, Elem<T>::mul2(w0, v[i][0].x))));
            o.y = Elem<T>::fma2p(w3, v[i][3].y, Elem<T>::fma2p(w2_, v[i][2].y, Elem<T>::fma2p(w1, v[i][1].y, Elem<T>::mul2(w0, v[i][0].y))));
            o.z = Elem<T>::fma2p(w3, v[i][3].z, Elem<T>::fma2p(w2_, v[i][2].z, Elem<T>::fma2p(w1, v[i][1].z, Elem<T>::mul2(w0, v[i][0].z))));
            o.w = Elem<T>::fma2p(w3, v[i][3].w, Elem<T>::fma2p(w2_, v[i][2].w, Elem<T>::fma2p(w1, v[i][1].w, Elem<T>::mul2(w0, v[i][0].w))));
          } else {
          unsigned long long acc[4] = {0ull, 0ull, 0ull, 0ull};   // 8 channels as 4 packed fp32 pairs (FFMA2)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t u[4] = {v[i][q].x, v[i][q].y, v[i][q].z, v[i][q].w};
            const unsigned long long w2 = pack2(wv[q], wv[q]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 f = Elem<T>::up(u[k]);
              acc[k] = fma2(w2, pack2(f.x, f.y), acc[k]);
            }
          }
          o.x = Elem<T>::pk(lo32(acc[0]), hi32(acc[0])); o.y = Elem<T>::pk(lo32(acc[1]), hi32(acc[1]));
          o.z = Elem<T>::pk(lo32(acc[2]), hi32(acc[2])); o.w = Elem<T>::pk(lo32(acc[3]), hi32(acc[3]));
          }
          const int prow = prow0 + 4 * i;
          *reinterpret_cast<uint4*>(a_tile + prow * ROW_BYTES + ((my_chunk ^ tc_swz<KB>(prow)) << 4)) = o;
        }
        fence_proxy_async();                  // generic-proxy stores -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int h = 0; h < SPLIT; ++h) mbar_arrive(&fullA[(q0 + h) % TC_STAGES]);
        }
      }
    }
    // ================= epilogue: TMEM -> registers -> NCHW =================
    mbar_wait(accum_full, 0u);
    tc_fence_after();
    const int lane_base = (warp & 3) * 32;
    const int col_half = warp >> 2;                           // four groups of 4 warps: a quarter of the columns each
    const int pix = pix0 + lane_base + lane;
    constexpr int COLS_PER_WARP = BN / (TC1_GATHER_WARPS / 4);
    // Full tiles of 16-byte aligned outputs: the 4 warps of a column group transpose 16 channels x 128 pixels through the (now
    // idle) pipeline stages and write each channel's 256 contiguous bytes with 16-byte vector stores - to `out` and to the peer
    // slots of the fused all-gather, where whole 256-byte runs instead of 64-byte ones make full NVLink packets.
    bool vec = sizeof(T) == 2 && pix0 + TC_BM <= HWo && (HWo % 8) == 0 && (reinterpret_cast<uintptr_t>(out) % 16) == 0;
    for (int d = 0; d < p.n_peer; ++d) vec = vec && (reinterpret_cast<uintptr_t>(p.peer_out[d]) % 16) == 0;
    if (vec) {
      constexpr int SLAB = 16 * TC_BM * 2;                    // 16 channels x 128 pixels, 2-byte elements
      unsigned char* est = stages + col_half * (2 * SLAB);    // two slabs per column group (alternating)
      const int tg = (warp & 3) * 32 + lane;                  // thread index inside the column group
#pragma unroll 1
      for (int c0 = 0, it = 0; c0 < COLS_PER_WARP; c0 += 16, ++it) {
        const int col = col_half * COLS_PER_WARP + c0;
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)col, r);
        T* slab = reinterpret_cast<T*>(est + (it & 1) * SLAB);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float bv = bias ? to_acc(bias[nt * BN + col + j]) : 0.f;
          slab[j * TC_BM + tg] = from_acc<T, float>(__uint_as_float(r[j]) + bv);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(2 + col_half) : "memory");
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int idx = tg + 128 * h, ch = idx >> 4, seg = idx & 15;
          const uint4 q = *reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(slab) + ch * (TC_BM * 2) + seg * 16);
          const int64_t eoff = (((int64_t)b * p.c_out + nt * BN + col + ch) * HWo + pix0) * 2 + seg * 16;      // bytes
          *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(out) + eoff) = q;
          for (int d = 0; d < p.n_peer; ++d) *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(p.peer_out[d]) + eoff) = q;
        }
      }
    } else {
#pragma unroll 1
      for (int c0 = 0; c0 < COLS_PER_WARP; c0 += 16) {
        const int col = col_half * COLS_PER_WARP + c0;
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)col, r);
        if (pix < HWo) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int co = nt * BN + col + j;
            const float bv = bias ? to_acc(bias[co]) : 0.f;
            const T v = from_acc<T, float>(__uint_as_float(r[j]) + bv);
            const int64_t idx = ((int64_t)b * p.c_out + co) * HWo + pix;
            out[idx] = v;
            for (int d = 0; d < p.n_peer; ++d) reinterpret_cast<T*>(p.peer_out[d])[idx] = v;     // fused all-gather: peer slots
          }
        }
      }
    }
    tc_fence_before();
  } else if (warp == TC1_GATHER_WARPS) {
    // ================= weight tiles: one bulk copy per stage =================
    if (lane == 0) {
      const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(wpacked) + (int64_t)nt * n_q * B_BYTES;
      for (int slab = 0; slab < n_q; ++slab) {
        const int st = slab % TC_STAGES;
        const uint32_t ph = (uint32_t)(slab / TC_STAGES) & 1u;
        mbar_wait(&empty[st], ph ^ 1u);
        mbar_expect_tx(&fullB[st], (uint32_t)B_BYTES);
        bulk_g2s(stages + st * STAGE_BYTES + TC_A_BYTES, wsrc + (int64_t)slab * B_BYTES, (uint32_t)B_BYTES, &fullB[st]);
      }
    }
  } else {
    // ================= MMA issuer =================
    if (lane == 0) {
      // cute::UMMA::InstrDescriptor: c_format F32 [4,6) | a_format [7,10) | b_format [10,13) | K-major A,B |
      // n_dim = N>>3 [17,23) | m_dim = M>>4 [24,29)
      constexpr int MMA_N = BN > 256 ? 256 : BN;
      const uint32_t idesc = (1u << 4) | (Elem<T>::kFmt << 7) | (Elem<T>::kFmt << 10) | ((uint32_t)(MMA_N >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      for (int slab = 0; slab < n_q; ++slab) {
        const int st = slab % TC_STAGES;
        const uint32_t ph = (uint32_t)(slab / TC_STAGES) & 1u;
        mbar_wait(&fullA[st], ph);
        mbar_wait(&fullB[st], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(stages + st * STAGE_BYTES);
        const uint32_t b_addr = a_addr + TC_A_BYTES;
#pragma unroll
        for (int k = 0; k < KB / 16; ++k) {
          umma_f16(tmem_base, smem_desc_k<KB>(a_addr + k * 32), smem_desc_k<KB>(b_addr + k * 32), idesc, (slab | k) ? 1u : 0u);
          if constexpr (BN > 256)       // second accumulator: output channels [256, 512) -> TMEM columns [256, 512)
            umma_f16(tmem_base + 256u, smem_desc_k<KB>(a_addr + k * 32), smem_desc_k<KB>(b_addr + 256 * ROW_BYTES + k * 32), idesc,
                     (slab | k) ? 1u : 0u);
        }
        umma_commit(&empty[st]);               // stage reusable once these MMAs have read it
      }
      umma_commit(accum_full);                 // all MMAs complete -> epilogue may read TMEM
    }
  }
  __syncthreads();
  if (warp == TC1_GATHER_WARPS + 1) { tc_fence_after(); tmem_dealloc(tmem_base, BN); }
}


// =================================================================================================
// CTA-pair variant (cta_group::2): a 2-CTA cluster computes a 256-pixel x 512-channel tile.
//   * each CTA gathers ITS 128 pixels (A rows) and loads HALF of the weight rows of every stage;
//     the leader CTA issues tcgen05.mma.cta_group::2 (M = 256, N = 256, two accumulators), each SM's
//     tensor core reads A and B-half from its own shared memory: per SM the operand reads drop from
//     96 to 64 B/cycle and the weight bytes written per stage halve — the single-CTA form saturates the
//     128 B/cycle shared-memory port (profiles/deform_conv2d_r1.md);
//   * synchronisation: the peer's gather warps arrive REMOTELY on the leader's fullA barrier; each
//     CTA's weight copy completes on its own fullB and the peer relays that to the leader's peerB;
//     tcgen05.commit multicasts to the empty / accum_full barriers of both CTAs.
// K depth 64 (SWIZZLE_128B), 3 stages of (16 KB A + 32 KB B-half) per CTA.
// =================================================================================================
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAITC_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONEC_%=;\n\t"
      "bra WAITC_%=;\n\t"
      "DONEC_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_c, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_c), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {   // arrives on `bar` of BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// weights for the CTA pair: per (cout tile of 512, rank r, slab q) a [256 rows][64 k] SWIZZLE_128B image;
// row rr = j*128 + i  <->  output channel nt*512 + j*256 + r*128 + i   (j = accumulator, r = CTA rank)
template <typename T>
__global__ void __launch_bounds__(256)
pack_weights2_kernel(const T* __restrict__ w, T* __restrict__ packed, int Cout, int Cin, int KK) {
  const int64_t total = (int64_t)Cout * Cin * KK;
  const int n_q = (Cin / 64) * KK;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int tap = (int)(e % KK);
    const int ci = (int)((e / KK) % Cin);
    const int co = (int)(e / KK / Cin);
    const int nt = co / 512, c5 = co % 512;
    const int j = c5 / 256, r = (c5 % 256) / 128, i = c5 % 128;
    const int rr = j * 128 + i;
    const int cslab = ci / 64, kc = ci % 64;
    const int q = cslab * KK + tap;
    const int64_t tile_base = (((int64_t)nt * 2 + r) * n_q + q) * 256 * 64;
    const int off_bytes = rr * 128 + (((kc >> 3) ^ (rr & 7)) << 4) + ((kc & 7) << 1);
    packed[tile_base + (off_bytes >> 1)] = w[e];
  }
}

constexpr int TC2_STAGES = 3;

template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
deform_conv2d_tc2_kernel(const T* __restrict__ nhwc, const T* __restrict__ wpacked, const T* __restrict__ offset,
                         const T* __restrict__ mask, const T* __restrict__ bias, T* __restrict__ out, DcnParams p,
                         int total_tiles) {
  constexpr int KB = 64, ROW_BYTES = 128;
  constexpr int A_BYTES = TC_BM * ROW_BYTES;            // 16 KB
  constexpr int B_BYTES = 256 * ROW_BYTES;              // 32 KB: this CTA's half of both accumulators' weights
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* stages = smem;
  uint64_t* fullA = reinterpret_cast<uint64_t*>(stages + TC2_STAGES * STAGE_BYTES);   // leader: 16 arrivals (8 + 8 remote)
  uint64_t* fullB = fullA + TC2_STAGES;                 // local weight copy (tx)
  uint64_t* peerB = fullB + TC2_STAGES;                 // leader: the peer's weight copy has landed
  uint64_t* empty = peerB + TC2_STAGES;                 // multicast commit
  uint64_t* accum_full = empty + TC2_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_full + 1);
  TcEnt* tab = reinterpret_cast<TcEnt*>(stages + ((TC2_STAGES * STAGE_BYTES + (4 * TC2_STAGES + 1) * 8 + 16 + 31) & ~31));

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int KK = p.kh * p.kw;
  const int HWo = p.out_h * p.out_w, HWi = p.in_h * p.in_w;
  const int tiles_per_img = ceil_div(HWo, TC_BM);
  const int tile = blockIdx.x;
  const bool live = tile < total_tiles;                 // the grid is padded to an even number of tiles
  const int b = live ? tile / tiles_per_img : 0;
  const int pix0 = live ? (tile % tiles_per_img) * TC_BM : HWo;
  const int nt = blockIdx.y;
  const int c_per_off = p.c_in / p.offset_groups;
  const int slabs_per_og = (c_per_off / 64) * KK;
  const int n_q = (p.c_in / 64) * KK;

  if (tid == 0) {
    for (int s = 0; s < TC2_STAGES; ++s) {
      mbar_init(&fullA[s], 2 * TC_GATHER_WARPS);
      mbar_init(&fullB[s], 1);
      mbar_init(&peerB[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(accum_full, 1);
    mbar_fence_init();
  }
  if (warp == TC_GATHER_WARPS + 1) tmem_alloc2(tmem_slot, 512);   // same warp id in both CTAs
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                   // barriers of both CTAs are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < TC_GATHER_WARPS) {
    const int cchunk = lane & 7, pq = lane >> 3;
    const int prow0 = warp * 16 + pq;
    const T* __restrict__ in_b = nhwc + (int64_t)b * HWi * p.c_in;
    int slab = 0;
    for (int og = 0; og < p.offset_groups; ++og) {
      asm volatile("bar.sync 1, %0;" ::"n"(TC_GATHER_THREADS));
      const T* __restrict__ off_b = offset + ((int64_t)b * p.offset_groups + og) * 2 * KK * HWo;
      const T* __restrict__ msk_b = p.use_mask ? mask + ((int64_t)b * p.offset_groups + og) * KK * HWo : nullptr;
      for (int e = tid; e < KK * TC_BM; e += TC_GATHER_THREADS) {
        const int tap = e / TC_BM, px = e - tap * TC_BM;
        const int pix = pix0 + px;
        TcEnt se;
#pragma unroll
        for (int q = 0; q < 4; ++q) { se.o[q] = 0; se.w[q] = 0.f; }
        if (pix < HWo) {
          const int oy = pix / p.out_w, ox = pix - oy * p.out_w;
          const int i = tap / p.kw, j = tap - i * p.kw;
          const float oh = to_acc(off_b[(int64_t)(2 * tap) * HWo + pix]);
          const float ow = to_acc(off_b[(int64_t)(2 * tap + 1) * HWo + pix]);
          const float mv = p.use_mask ? to_acc(msk_b[(int64_t)tap * HWo + pix]) : 1.f;
          const float y = add_rn((float)(oy * p.stride_h - p.pad_h + i * p.dil_h), oh);
          const float x = add_rn((float)(ox * p.stride_w - p.pad_w + j * p.dil_w), ow);
          if (!(y <= -1.f || (float)p.in_h <= y || x <= -1.f || (float)p.in_w <= x)) {
            const int hl = (int)floorf(y), wl = (int)floorf(x);
            const int hh_i = hl + 1, wh_i = wl + 1;
            const float lh = y - (float)hl, lw = x - (float)wl;
            const float hh = 1.f - lh, hw = 1.f - lw;
            const bool t0 = hl >= 0, t1 = hh_i <= p.in_h - 1, l0 = wl >= 0, l1 = wh_i <= p.in_w - 1;
            const int hlc = max(hl, 0), hhc = min(hh_i, p.in_h - 1), wlc = max(wl, 0), whc = min(wh_i, p.in_w - 1);
            se.o[0] = (hlc * p.in_w + wlc) * p.c_in; se.w[0] = (t0 && l0) ? mv * (hh * hw) : 0.f;
            se.o[1] = (hlc * p.in_w + whc) * p.c_in; se.w[1] = (t0 && l1) ? mv * (hh * lw) : 0.f;
            se.o[2] = (hhc * p.in_w + wlc) * p.c_in; se.w[2] = (t1 && l0) ? mv * (lh * hw) : 0.f;
            se.o[3] = (hhc * p.in_w + whc) * p.c_in; se.w[3] = (t1 && l1) ? mv * (lh * lw) : 0.f;
          }
        }
        tab[e] = se;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(TC_GATHER_THREADS));
      for (int sl = 0; sl < slabs_per_og; ++sl, ++slab) {
        const int cs_local = sl / KK, tap = sl - cs_local * KK;
        const T* __restrict__ in_c = in_b + og * c_per_off + cs_local * 64 + cchunk * 8;
        const int st = slab % TC2_STAGES;
        const uint32_t ph = (uint32_t)(slab / TC2_STAGES) & 1u;
        uint4 v[4][4];
        float4 wq[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const TcEnt* se = tab + tap * TC_BM + prow0 + 4 * i;
          const int4 o = *reinterpret_cast<const int4*>(se->o);
          wq[i] = *reinterpret_cast<const float4*>(se->w);
          v[i][0] = __ldg(reinterpret_cast<const uint4*>(in_c + o.x));
          v[i][1] = __ldg(reinterpret_cast<const uint4*>(in_c + o.y));
          v[i][2] = __ldg(reinterpret_cast<const uint4*>(in_c + o.z));
          v[i][3] = __ldg(reinterpret_cast<const uint4*>(in_c + o.w));
        }
        mbar_wait(&empty[st], ph ^ 1u);
        unsigned char* a_tile = stages + st * STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float wv[4] = {wq[i].x, wq[i].y, wq[i].z, wq[i].w};
          unsigned long long acc[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t u[4] = {v[i][q].x, v[i][q].y, v[i][q].z, v[i][q].w};
            const unsigned long long w2 = pack2(wv[q], wv[q]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 f = Elem<T>::up(u[k]);
              acc[k] = fma2(w2, pack2(f.x, f.y), acc[k]);
            }
          }
          uint4 o;
          o.x = Elem<T>::pk(lo32(acc[0]), hi32(acc[0])); o.y = Elem<T>::pk(lo32(acc[1]), hi32(acc[1]));
          o.z = Elem<T>::pk(lo32(acc[2]), hi32(acc[2])); o.w = Elem<T>::pk(lo32(acc[3]), hi32(acc[3]));
          const int prow = prow0 + 4 * i;
          *reinterpret_cast<uint4*>(a_tile + prow * ROW_BYTES + ((cchunk ^ (prow & 7)) << 4)) = o;
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(&fullA[st]); else mbar_arrive_remote(&fullA[st], 0u);
        }
      }
    }
    // ---- epilogue: this CTA's 128 pixel rows x 512 channels ----
    mbar_wait_cluster(accum_full, 0u);
    tc_fence_after();
    const int lane_base = (warp & 3) * 32;
    const int col_half = warp >> 2;
    const int pix = pix0 + lane_base + lane;
#pragma unroll 1
    for (int c0 = 0; c0 < 256; c0 += 16) {
      const int col = col_half * 256 + c0;
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)col, r);
      if (live && pix < HWo) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int co = nt * 512 + col + j;
          const float bv = bias ? to_acc(bias[co]) : 0.f;
          out[((int64_t)b * p.c_out + co) * HWo + pix] = from_acc<T, float>(__uint_as_float(r[j]) + bv);
        }
      }
    }
    tc_fence_before();
  } else if (warp == TC_GATHER_WARPS) {
    // ---- weights: lane 0 streams this CTA's half tiles; on the peer, lane 1 relays "landed" to the leader ----
    if (lane == 0) {
      const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(wpacked) + ((int64_t)nt * 2 + rank) * n_q * B_BYTES;
      for (int q = 0; q < n_q; ++q) {
        const int st = q % TC2_STAGES;
        const uint32_t ph = (uint32_t)(q / TC2_STAGES) & 1u;
        mbar_wait(&empty[st], ph ^ 1u);
        mbar_expect_tx(&fullB[st], (uint32_t)B_BYTES);
        bulk_g2s(stages + st * STAGE_BYTES + A_BYTES, wsrc + (int64_t)q * B_BYTES, (uint32_t)B_BYTES, &fullB[st]);
      }
    } else if (lane == 1 && !leader) {
      for (int q = 0; q < n_q; ++q) {
        const int st = q % TC2_STAGES;
        const uint32_t ph = (uint32_t)(q / TC2_STAGES) & 1u;
        mbar_wait(&fullB[st], ph);
        mbar_arrive_remote(&peerB[st], 0u);
      }
    }
  } else {
    // ---- MMA issuer: leader CTA only ----
    if (lane == 0 && leader) {
      const uint32_t idesc = (1u << 4) | (Elem<T>::kFmt << 7) | (Elem<T>::kFmt << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      for (int q = 0; q < n_q; ++q) {
        const int st = q % TC2_STAGES;
        const uint32_t ph = (uint32_t)(q / TC2_STAGES) & 1u;
        mbar_wait_cluster(&fullA[st], ph);
        mbar_wait(&fullB[st], ph);
        mbar_wait_cluster(&peerB[st], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(stages + st * STAGE_BYTES);
        const uint32_t b_addr = a_addr + A_BYTES;
#pragma unroll
        for (int k = 0; k < KB / 16; ++k) {
          umma2_f16(tmem_base, smem_desc_k<KB>(a_addr + k * 32), smem_desc_k<KB>(b_addr + k * 32), idesc, (q | k) ? 1u : 0u);
          umma2_f16(tmem_base + 256u, smem_desc_k<KB>(a_addr + k * 32), smem_desc_k<KB>(b_addr + 128 * ROW_BYTES + k * 32), idesc,
                    (q | k) ? 1u : 0u);
        }
        umma2_commit_mc(&empty[st]);
      }
      umma2_commit_mc(accum_full);
    }
  }
  __syncthreads();
  cluster_sync_all();                                   // nobody leaves (or frees TMEM) while the pair is still in use
  if (warp == TC_GATHER_WARPS + 1) { tc_fence_after(); tmem_dealloc2(tmem_base, 512); }
}

// =================================================================================================
// fp32 inputs on the tensor core: three-way bf16 split (bf16x3).
// A float v is v1 + v2 + v3 with v1 = bf16(v), v2 = bf16(v - v1), v3 = bf16(v - v1 - v2) (8 + 8 + 8 mantissa bits); the
// product a*b is a1b1 + (a1b2 + a2b1) + (a2b2 + a1b3 + a3b1) + O(2^-24): SIX kind::f16 MMAs per K step into the same fp32
// TMEM accumulator reproduce the fp32 result to ~1e-7 relative per product - inside the 1e-5 budget of the fp32 rows,
// at 6x the bf16 tensor time, which is still several times faster than a SIMT fp32 implicit GEMM (or the reference's
// im2col + SGEMM).  Same structure as deform_conv2d_tc_kernel: M = 128 pixels, N = BN couts, K step 32 channels
// (SWIZZLE_64B); a stage holds A1 A2 A3 (8 KB each) and B1 B2 B3 (BN x 64 B each); the gather reads a channels-last
// fp32 staging copy (one 128-byte line = 32 channels per pixel corner), blends in fp32 and writes the three splits.
// ACCUMULATION: the tensor core adds into its fp32 accumulator with truncation (measured: ~one ulp of the accumulator
// lost per MMA instruction, a bias that grows linearly with the number of MMAs - 8e-5 absolute after 864 MMAs into one
// accumulator).  So (1) the five correction terms go to their OWN accumulator (its magnitude is 2^-8 of the result, so its
// truncation is invisible) and (2) the a1 b1 terms rotate over THREE accumulators by K step; the epilogue adds the four
// TMEM regions in registers with round-to-nearest.  BN = 128: 3 + 1 accumulators x 128 columns = all 512 TMEM columns.
// =================================================================================================
constexpr int T3_KB = 32, T3_STAGES = 3, T3_MAIN = 3;
constexpr int T3_ROW = 2 * T3_KB;                 // 64-byte tile rows
constexpr int T3_A = TC_BM * T3_ROW;              // 8 KB per A split

__device__ __forceinline__ void split3(float v, __nv_bfloat16& a, __nv_bfloat16& b, __nv_bfloat16& c) {
  a = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(a);      // exact: the residual has at most 16 significant bits
  b = __float2bfloat16_rn(r1);
  c = __float2bfloat16_rn(r1 - __bfloat162float(b));
}

// weights [Cout][Cin][KK] fp32 -> per (n tile, stage q = cslab32 * KK + tap): B1 | B2 | B3 swizzled tiles of BN x 32
__global__ void __launch_bounds__(256)
pack_weights3_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ packed, int Cout, int Cin, int KK, int BN) {
  const int64_t total = (int64_t)Cout * Cin * KK;
  const int n_q = (Cin / T3_KB) * KK;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int tap = (int)(e % KK);
    const int ci = (int)((e / KK) % Cin);
    const int co = (int)(e / KK / Cin);
    const int nt = co / BN, r = co % BN;
    const int cslab = ci / T3_KB, kc = ci % T3_KB;
    const int q = cslab * KK + tap;
    const int64_t stage_base = ((int64_t)nt * n_q + q) * 3 * BN * T3_KB;            // elements
    const int off = (r * T3_ROW + (((kc >> 3) ^ tc_swz<T3_KB>(r)) << 4) + ((kc & 7) << 1)) >> 1;
    __nv_bfloat16 b1, b2, b3;
    split3(w[e], b1, b2, b3);
    packed[stage_base + off] = b1;
    packed[stage_base + (int64_t)BN * T3_KB + off] = b2;
    packed[stage_base + (int64_t)2 * BN * T3_KB + off] = b3;
  }
}

template <int BN>
__global__ void __launch_bounds__(TC1_THREADS, 1)
deform_conv2d_tc3_kernel(const float* __restrict__ nhwc, const __nv_bfloat16* __restrict__ wpacked, const float* __restrict__ offset,
                         const float* __restrict__ mask, const float* __restrict__ bias, float* __restrict__ out, DcnParams p) {
  constexpr int B_BYTES = BN * T3_ROW;                    // one B split
  constexpr int STAGE_BYTES = 3 * T3_A + 3 * B_BYTES;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* stages = smem;
  uint64_t* fullA = reinterpret_cast<uint64_t*>(stages + T3_STAGES * STAGE_BYTES);
  uint64_t* fullB = fullA + T3_STAGES;
  uint64_t* empty = fullB + T3_STAGES;
  uint64_t* accum_full = empty + T3_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_full + 1);
  TcEnt* tab = reinterpret_cast<TcEnt*>(stages + ((T3_STAGES * STAGE_BYTES + (3 * T3_STAGES + 1) * 8 + 16 + 31) & ~31));

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int KK = p.kh * p.kw;
  const int HWo = p.out_h * p.out_w, HWi = p.in_h * p.in_w;
  const int tiles_per_img = ceil_div(HWo, TC_BM);
  const int b = blockIdx.x / tiles_per_img;
  const int pix0 = (blockIdx.x % tiles_per_img) * TC_BM;
  const int nt = blockIdx.y;
  const int c_per_off = p.c_in / p.offset_groups;
  const int slabs_per_og = (c_per_off / T3_KB) * KK;      // 32-channel gather steps per offset group
  const int n_q = (p.c_in / T3_KB) * KK;                  // stages consumed per tile

  if (tid == 0) {
    for (int s = 0; s < T3_STAGES; ++s) { mbar_init(&fullA[s], TC_GATHER_WARPS); mbar_init(&fullB[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(accum_full, 1);
    mbar_fence_init();
  }
  static_assert(BN * (T3_MAIN + 1) <= 512, "3 main + 1 correction accumulator must fit TMEM");
  if (warp == TC1_GATHER_WARPS + 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < TC1_GATHER_WARPS) {
    // two groups of 8 gather warps take alternate 32-channel steps
    const int group = warp >> 3, wg = warp & 7;
    const int cchunk = lane & 7, pq = lane >> 3;           // lane -> (pixel sub-index, 4-channel chunk of the 32-channel line)
    const int prow0 = wg * 16 + pq;
    const float* __restrict__ in_b = nhwc + (int64_t)b * HWi * p.c_in;
    for (int og = 0; og < p.offset_groups; ++og) {
      asm volatile("bar.sync 1, %0;" ::"n"(TC1_GATHER_THREADS));
      const float* __restrict__ off_b = offset + ((int64_t)b * p.offset_groups + og) * 2 * KK * HWo;
      const float* __restrict__ msk_b = p.use_mask ? mask + ((int64_t)b * p.offset_groups + og) * KK * HWo : nullptr;
      for (int e = tid; e < KK * TC_BM; e += TC1_GATHER_THREADS) {
        const int tap = e / TC_BM, px = e - tap * TC_BM;
        const int pix = pix0 + px;
        TcEnt se;
#pragma unroll
        for (int q = 0; q < 4; ++q) { se.o[q] = 0; se.w[q] = 0.f; }
        if (pix < HWo) {
          const int oy = pix / p.out_w, ox = pix - oy * p.out_w;
          const int i = tap / p.kw, j = tap - i * p.kw;
          const float oh = off_b[(int64_t)(2 * tap) * HWo + pix];
          const float ow = off_b[(int64_t)(2 * tap + 1) * HWo + pix];
          const float mv = p.use_mask ? msk_b[(int64_t)tap * HWo + pix] : 1.f;
          const float y = add_rn((float)(oy * p.stride_h - p.pad_h + i * p.dil_h), oh);
          const float x = add_rn((float)(ox * p.stride_w - p.pad_w + j * p.dil_w), ow);
          if (!(y <= -1.f || (float)p.in_h <= y || x <= -1.f || (float)p.in_w <= x)) {
            const int hl = (int)floorf(y), wl = (int)floorf(x);
            const int hh_i = hl + 1, wh_i = wl + 1;
            const float lh = y - (float)hl, lw = x - (float)wl;
            const float hh = 1.f - lh, hw = 1.f - lw;
            const bool t0 = hl >= 0, t1 = hh_i <= p.in_h - 1, l0 = wl >= 0, l1 = wh_i <= p.in_w - 1;
            const int hlc = max(hl, 0), hhc = min(hh_i, p.in_h - 1), wlc = max(wl, 0), whc = min(wh_i, p.in_w - 1);
            se.o[0] = (hlc * p.in_w + wlc) * p.c_in * 4; se.w[0] = (t0 && l0) ? mv * (hh * hw) : 0.f;
            se.o[1] = (hlc * p.in_w + whc) * p.c_in * 4; se.w[1] = (t0 && l1) ? mv * (hh * lw) : 0.f;
            se.o[2] = (hhc * p.in_w + wlc) * p.c_in * 4; se.w[2] = (t1 && l0) ? mv * (lh * hw) : 0.f;
            se.o[3] = (hhc * p.in_w + whc) * p.c_in * 4; se.w[3] = (t1 && l1) ? mv * (lh * lw) : 0.f;
          }
        }
        tab[e] = se;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(TC1_GATHER_THREADS));
      const int slab_base = og * slabs_per_og;
      for (int sl = (slab_base + group) & 1; sl < slabs_per_og; sl += 2) {
        const int q = slab_base + sl;
        const int cs_local = sl / KK, tap = sl - cs_local * KK;
        const char* __restrict__ in_c = reinterpret_cast<const char*>(in_b + og * c_per_off + cs_local * T3_KB);
        const uint32_t lane_off = (uint32_t)cchunk * 16u;
        float4 v[4][4];
        float4 wq[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const TcEnt* se = tab + tap * TC_BM + prow0 + 4 * i;
          const uint4 o = *reinterpret_cast<const uint4*>(se->o);
          wq[i] = *reinterpret_cast<const float4*>(se->w);
          v[i][0] = __ldg(reinterpret_cast<const float4*>(in_c + (o.x + lane_off)));
          v[i][1] = __ldg(reinterpret_cast<const float4*>(in_c + (o.y + lane_off)));
          v[i][2] = __ldg(reinterpret_cast<const float4*>(in_c + (o.z + lane_off)));
          v[i][3] = __ldg(reinterpret_cast<const float4*>(in_c + (o.w + lane_off)));
        }
        mbar_wait(&empty[q % T3_STAGES], ((uint32_t)(q / T3_STAGES) & 1u) ^ 1u);
        unsigned char* a_tile = stages + (q % T3_STAGES) * STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          // fp32 blend in the reference's tap order (w1 v1 + w2 v2 + w3 v3 + w4 v4, deform_conv2d_kernel.cu:128-133)
          float r[4];
          r[0] = wq[i].x * v[i][0].x + wq[i].y * v[i][1].x + wq[i].z * v[i][2].x + wq[i].w * v[i][3].x;
          r[1] = wq[i].x * v[i][0].y + wq[i].y * v[i][1].y + wq[i].z * v[i][2].y + wq[i].w * v[i][3].y;
          r[2] = wq[i].x * v[i][0].z + wq[i].y * v[i][1].z + wq[i].z * v[i][2].z + wq[i].w * v[i][3].z;
          r[3] = wq[i].x * v[i][0].w + wq[i].y * v[i][1].w + wq[i].z * v[i][2].w + wq[i].w * v[i][3].w;
          __nv_bfloat16 s1[4], s2[4], s3[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) split3(r[k], s1[k], s2[k], s3[k]);
          const int prow = prow0 + 4 * i;
          // this lane's 4 channels are half of a 16-byte chunk: chunk (cchunk >> 1), byte half (cchunk & 1)
          const int boff = prow * T3_ROW + ((((cchunk >> 1) ^ tc_swz<T3_KB>(prow)) << 4) | ((cchunk & 1) << 3));
          *reinterpret_cast<uint2*>(a_tile + boff) = *reinterpret_cast<const uint2*>(s1);
          *reinterpret_cast<uint2*>(a_tile + T3_A + boff) = *reinterpret_cast<const uint2*>(s2);
          *reinterpret_cast<uint2*>(a_tile + 2 * T3_A + boff) = *reinterpret_cast<const uint2*>(s3);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&fullA[q % T3_STAGES]);
      }
    }
    // ================= epilogue: TMEM -> registers -> NCHW fp32 =================
    mbar_wait(accum_full, 0u);
    tc_fence_after();
    const int lane_base = (warp & 3) * 32;
    const int col_q = warp >> 2;
    const int pix = pix0 + lane_base + lane;
    constexpr int COLS_PER_WARP = BN / (TC1_GATHER_WARPS / 4);
#pragma unroll 1
    for (int c0 = 0; c0 < COLS_PER_WARP; c0 += 16) {
      const int col = col_q * COLS_PER_WARP + c0;
      uint32_t r0[16], r1[16], r2[16], rs[16];
      const uint32_t ta = tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)col;
      tmem_ld16(ta, r0);
      tmem_ld16(ta + BN, r1);
      tmem_ld16(ta + 2 * BN, r2);
      tmem_ld16(ta + 3 * BN, rs);
      if (pix < HWo) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int co = nt * BN + col + j;
          const float main = (n_q > 2 ? __uint_as_float(r2[j]) : 0.f) + ((n_q > 1 ? __uint_as_float(r1[j]) : 0.f) + __uint_as_float(r0[j]));
          out[((int64_t)b * p.c_out + co) * HWo + pix] = (main + __uint_as_float(rs[j])) + (bias ? bias[co] : 0.f);
        }
      }
    }
    tc_fence_before();
  } else if (warp == TC1_GATHER_WARPS) {
    if (lane == 0) {
      const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(wpacked) + (int64_t)nt * n_q * 3 * B_BYTES;
      for (int q = 0; q < n_q; ++q) {
        const int st = q % T3_STAGES;
        const uint32_t ph = (uint32_t)(q / T3_STAGES) & 1u;
        mbar_wait(&empty[st], ph ^ 1u);
        mbar_expect_tx(&fullB[st], (uint32_t)(3 * B_BYTES));
        bulk_g2s(stages + st * STAGE_BYTES + 3 * T3_A, wsrc + (int64_t)q * 3 * B_BYTES, (uint32_t)(3 * B_BYTES), &fullB[st]);
      }
    }
  } else {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);   // bf16 x bf16 -> fp32
      for (int q = 0; q < n_q; ++q) {
        const int st = q % T3_STAGES;
        const uint32_t ph = (uint32_t)(q / T3_STAGES) & 1u;
        mbar_wait(&fullA[st], ph);
        mbar_wait(&fullB[st], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(stages + st * STAGE_BYTES);
        const uint32_t b_addr = a_addr + 3 * T3_A;
        // correction terms (a3b1, a1b3, a2b2, a2b1, a1b2) -> their own accumulator at column 3 * BN
        constexpr int ia[5] = {2, 0, 1, 1, 0}, ib[5] = {0, 2, 1, 0, 1};
#pragma unroll
        for (int t = 0; t < 5; ++t) {
#pragma unroll
          for (int k = 0; k < T3_KB / 16; ++k)
            umma_f16(tmem_base + 3u * BN, smem_desc_k<T3_KB>(a_addr + ia[t] * T3_A + k * 32),
                     smem_desc_k<T3_KB>(b_addr + ib[t] * B_BYTES + k * 32), idesc, (q | t | k) ? 1u : 0u);
        }
        // a1 b1 -> main accumulator q mod 3 (first touch of each starts from zero)
        const uint32_t main_col = (uint32_t)(q % T3_MAIN) * BN;
#pragma unroll
        for (int k = 0; k < T3_KB / 16; ++k)
          umma_f16(tmem_base + main_col, smem_desc_k<T3_KB>(a_addr + k * 32), smem_desc_k<T3_KB>(b_addr + k * 32), idesc,
                   (q >= T3_MAIN || k) ? 1u : 0u);
        umma_commit(&empty[st]);
      }
      umma_commit(accum_full);
    }
  }
  __syncthreads();
  if (warp == TC1_GATHER_WARPS + 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

size_t tc3_smem_bytes(int BN, int KK) {
  return (size_t)T3_STAGES * (3 * T3_A + 3 * BN * T3_ROW) + 128 + (size_t)KK * TC_BM * sizeof(TcEnt) + 1024;
}
int tc3_pick_bn(const DcnParams& p) {
  const int KK = p.kh * p.kw;
  return (p.c_out % 128 == 0 && tc3_smem_bytes(128, KK) <= (size_t)max_smem_optin()) ? 128 : 0;
}
bool tc3_eligible(int dtype, const DcnParams& p) {
  if (dtype != VB200_F32 || p.groups != 1) return false;
  if (p.c_in % p.offset_groups != 0 || (p.c_in / p.offset_groups) % T3_KB != 0) return false;
  if (p.c_out % 128 != 0 || tc3_pick_bn(p) == 0) return false;
  if ((int64_t)p.in_h * p.in_w * p.c_in * 4 >= (1ll << 31)) return false;      // 32-bit byte offsets into one image
  const char* env = env_override(ENV_DCN_PATH);
  if (env && env[0] == 's') return false;
  return true;
}

size_t tc2_smem_bytes(int KK) {
  return (size_t)TC2_STAGES * (TC_BM + 256) * 128 + 256 + (size_t)KK * TC_BM * sizeof(TcEnt) + 1024;
}
bool tc2_enabled(const DcnParams& p) {
  const char* env = env_override(ENV_DCN_CTA2);
  if (!(env && env[0] == '1')) return false;
  return p.c_out % 512 == 0 && tc2_smem_bytes(p.kh * p.kw) <= (size_t)max_smem_optin();
}

// BN <= 256: K depth 64, 3 stages.  BN = 512: K depth 32, 4 stages (the 64 KB weight tile of a 64-deep
// stage leaves room for only 2 stages, which exposes the L2 latency of every refill).
constexpr int tc_kb(int BN) { return BN > 256 ? 32 : 64; }
// pipeline depth: BN <= 256 -> 3 x (16 + BN/8) KB; BN = 512 -> N x 40 KB, N = 4 by default
// (VB200_DCN_STAGES=3|4 overrides, for profiling: fewer stages leave more of the 228 KB to L1 — measured:
// no gain, profiles/deform_conv2d_r1.md).
// No 2-stage variant: a 64-channel gather step fills both K-32 stages, so each gather group would wait on stages whose
// previous round belongs to the other group and its own round before that; when its own previous step is still
// unconsumed, the empty barrier is two phases behind and its parity reads as "free" - the step overwrites live operands.
int tc_stages(int BN) {
  if (BN <= 256) return 3;
  const char* env = env_override(ENV_DCN_STAGES);
  const int n = env ? atoi(env) : 4;        // 4: each gather group owns its own pair of K-32 stages
  return n == 3 ? 3 : 4;
}
size_t tc_smem_bytes(int BN, int KK) {
  return (size_t)tc_stages(BN) * (TC_BM + BN) * 2 * tc_kb(BN) + 128 + (size_t)KK * TC_BM * sizeof(TcEnt) + 1024;
}
int tc_pick_bn(const DcnParams& p) {
  const char* env = env_override(ENV_DCN_BN);           // profiling override: 128 / 256 / 512
  const int KK = p.kh * p.kw;
  const int cands[3] = {512, 256, 128};
  for (int c = 0; c < 3; ++c) {
    const int bn = cands[c];
    if (env && atoi(env) != bn) continue;
    if (p.c_out % bn == 0 && tc_smem_bytes(bn, KK) <= (size_t)max_smem_optin()) return bn;
  }
  for (int c = 0; c < 3; ++c)
    if (p.c_out % cands[c] == 0 && tc_smem_bytes(cands[c], KK) <= (size_t)max_smem_optin()) return cands[c];
  return 0;
}

bool tc_eligible(int dtype, const DcnParams& p) {
  if (dtype != VB200_BF16 && dtype != VB200_F16) return false;
  if (p.groups != 1) return false;
  if (p.c_in % p.offset_groups != 0 || (p.c_in / p.offset_groups) % 64 != 0) return false;
  if (p.c_out % 128 != 0) return false;
  if (tc_pick_bn(p) == 0) return false;
  if ((int64_t)p.in_h * p.in_w * p.c_in >= (1ll << 30)) return false;      // 32-bit byte offsets into one image
  const char* env = env_override(ENV_DCN_PATH);
  if (env && env[0] == 's') return false;
  return true;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

template <typename T>
int pack_tc_weights(const void* weight, T* wpacked, const DcnParams& p, cudaStream_t st) {
  const int KK = p.kh * p.kw;
  if (tc2_enabled(p)) {
    pack_weights2_kernel<T><<<sm_count() * 4, 256, 0, st>>>((const T*)weight, wpacked, p.c_out, p.c_in, KK);
    return check_launch("pack_weights2_kernel");
  }
  const int BN = tc_pick_bn(p);
  if (tc_kb(512) == 32 && BN == 512)
    pack_weights_kernel<T, 32><<<sm_count() * 4, 256, 0, st>>>((const T*)weight, wpacked, p.c_out, p.c_in, KK, BN);
  else
    pack_weights_kernel<T, 64><<<sm_count() * 4, 256, 0, st>>>((const T*)weight, wpacked, p.c_out, p.c_in, KK, BN);
  return check_launch("pack_weights_kernel");
}

template <typename T>
int launch_tc(const void* input, const void* weight, const void* offset, const void* mask, const void* bias, void* out,
              const DcnParams& p_in, void* workspace, size_t workspace_bytes, cudaStream_t st, const DcnHints& hints) {
  DcnParams p = p_in;
  {
    // corner blend: fp32 FFMA2, or packed in the storage format (HFMA2: -5 % time).  Default: packed for fp16 (worst error 0.13 of
    // the 1e-2 bound on cfg4), fp32 for bf16 (the packed bf16 blend reaches 1.06 of the bound); VB200_DCN_BLEND=16|32 overrides.
    const char* env = env_override(ENV_DCN_BLEND);
    p.blend16 = env ? (env[0] == '1' && env[1] == '6') : (sizeof(T) == 2 && std::is_same<T, __half>::value);
  }
  const int KK = p.kh * p.kw, HWi = p.in_h * p.in_w, HWo = p.out_h * p.out_w;
  const size_t nhwc_bytes = hints.input_is_nhwc ? 0 : align256((size_t)p.batch * HWi * p.c_in * sizeof(T));
  const size_t w_bytes = hints.packed_weight ? 0 : align256((size_t)p.c_out * p.c_in * KK * sizeof(T));
  if (nhwc_bytes + w_bytes > 0 && (workspace == nullptr || workspace_bytes < nhwc_bytes + w_bytes || ((uintptr_t)workspace % 256) != 0))
    return 0;       // no usable workspace: the SIMT kernel serves the call (a C-ABI caller may pass none)
  T* nhwc = hints.input_is_nhwc ? (T*)const_cast<void*>(input) : (T*)workspace;
  T* wpacked = hints.packed_weight ? (T*)const_cast<void*>(hints.packed_weight) : (T*)((char*)workspace + nhwc_bytes);
  if (hints.input_is_nhwc) {
    if (((uintptr_t)input % 16) != 0) { set_error("deform_conv2d: channels-last input must be 16-byte aligned"); return VB200_EINVAL; }
  } else if (HWi % 2 == 0 && p.c_in % 64 == 0 && ((uintptr_t)input % 4) == 0) {
    dim3 tg((unsigned)ceil_div(HWi, 64), (unsigned)(p.c_in / 64), (unsigned)p.batch);
    nchw_to_nhwc64_kernel<T><<<tg, 256, 0, st>>>((const T*)input, nhwc, p.c_in, HWi);
  } else {
    dim3 tg((unsigned)ceil_div(HWi, 32), (unsigned)ceil_div(p.c_in, 32), (unsigned)p.batch);
    nchw_to_nhwc_kernel<T><<<tg, 256, 0, st>>>((const T*)input, nhwc, p.c_in, HWi);
  }
  int rc = hints.input_is_nhwc ? 0 : check_launch("nchw_to_nhwc_kernel");
  if (rc) return rc;
  if (!hints.packed_weight) {
    rc = pack_tc_weights<T>(weight, wpacked, p, st);
    if (rc) return rc;
  }
  if (tc2_enabled(p)) {
    const int total_tiles = p.batch * ceil_div(HWo, TC_BM);
    dim3 grid2((unsigned)((total_tiles + 1) & ~1), (unsigned)(p.c_out / 512));
    const size_t smem2 = tc2_smem_bytes(KK);
    VB200_CUDA_TRY(ensure_dyn_smem<deform_conv2d_tc2_kernel<T>>(smem2));
    deform_conv2d_tc2_kernel<T><<<grid2, TC_THREADS, smem2, st>>>(nhwc, wpacked, (const T*)offset, (const T*)mask,
                                                                  (const T*)bias, (T*)out, p, total_tiles);
    rc = check_launch("deform_conv2d_tc2_kernel");
    return rc ? rc : 1;
  }
  const int BN = tc_pick_bn(p);
  dim3 grid((unsigned)(p.batch * ceil_div(HWo, TC_BM)), (unsigned)(p.c_out / BN));
  const size_t smem = tc_smem_bytes(BN, KK);
  p.n_peer = hints.peer_out ? hints.n_peer : 0;
  for (int d = 0; d < p.n_peer; ++d) p.peer_out[d] = hints.peer_out[d];
  if (hints.peers_done) *hints.peers_done = true;
#define VB200_TC_LAUNCH(BN_, ST_)                                                                                         \
  {                                                                                                                       \
    VB200_CUDA_TRY(ensure_dyn_smem<deform_conv2d_tc_kernel<T, BN_, ST_, tc_kb(BN_)>>(smem));                         \
    deform_conv2d_tc_kernel<T, BN_, ST_, tc_kb(BN_)><<<grid, TC1_THREADS, smem, st>>>(                                    \
        nhwc, wpacked, (const T*)offset, (const T*)mask, (const T*)bias, (T*)out, p);                                     \
  }
  const int nst = tc_stages(BN);
  if (BN == 512) {
    if (nst == 4) VB200_TC_LAUNCH(512, 4) else VB200_TC_LAUNCH(512, 3)
  } else if (BN == 256) VB200_TC_LAUNCH(256, 3) else VB200_TC_LAUNCH(128, 3)
#undef VB200_TC_LAUNCH
  rc = check_launch("deform_conv2d_tc_kernel");
  return rc ? rc : 1;
}

}  // namespace

int launch_tc3(const void* input, const void* weight, const void* offset, const void* mask, const void* bias, void* out,
               const DcnParams& p, void* workspace, size_t workspace_bytes, cudaStream_t st, const DcnHints& hints) {
  const int KK = p.kh * p.kw, HWi = p.in_h * p.in_w, HWo = p.out_h * p.out_w;
  const size_t nhwc_bytes = hints.input_is_nhwc ? 0 : align256((size_t)p.batch * HWi * p.c_in * 4);
  const size_t w_bytes = hints.packed_weight ? 0 : align256((size_t)p.c_out * p.c_in * KK * 3 * 2);
  if (nhwc_bytes + w_bytes > 0 && (workspace == nullptr || workspace_bytes < nhwc_bytes + w_bytes || ((uintptr_t)workspace % 256) != 0))
    return 0;   // SIMT kernel serves the call
  float* nhwc = hints.input_is_nhwc ? (float*)const_cast<void*>(input) : (float*)workspace;
  __nv_bfloat16* wpacked = hints.packed_weight ? (__nv_bfloat16*)const_cast<void*>(hints.packed_weight) : (__nv_bfloat16*)((char*)workspace + nhwc_bytes);
  int rc = 0;
  if (!hints.input_is_nhwc) {
    dim3 tg((unsigned)ceil_div(HWi, 32), (unsigned)ceil_div(p.c_in, 32), (unsigned)p.batch);
    nchw_to_nhwc_kernel<float><<<tg, 256, 0, st>>>((const float*)input, nhwc, p.c_in, HWi);
    rc = check_launch("nchw_to_nhwc_kernel");
    if (rc) return rc;
  } else if (((uintptr_t)input % 16) != 0) { set_error("deform_conv2d: channels-last input must be 16-byte aligned"); return VB200_EINVAL; }
  const int BN = tc3_pick_bn(p);
  if (!hints.packed_weight) {
    pack_weights3_kernel<<<sm_count() * 4, 256, 0, st>>>((const float*)weight, wpacked, p.c_out, p.c_in, KK, BN);
    rc = check_launch("pack_weights3_kernel");
    if (rc) return rc;
  }
  dim3 grid((unsigned)(p.batch * ceil_div(HWo, TC_BM)), (unsigned)(p.c_out / BN));
  const size_t smem = tc3_smem_bytes(BN, KK);
  VB200_CUDA_TRY(ensure_dyn_smem<deform_conv2d_tc3_kernel<128>>(smem));
  deform_conv2d_tc3_kernel<128><<<grid, TC1_THREADS, smem, st>>>(nhwc, wpacked, (const float*)offset, (const float*)mask,
                                                                (const float*)bias, (float*)out, p);
  rc = check_launch("deform_conv2d_tc3_kernel");
  return rc ? rc : 1;
}

size_t deform_conv2d_tc_workspace(int dtype, const DcnParams& p) {
  if (tc3_eligible(dtype, p))
    return align256((size_t)p.batch * p.in_h * p.in_w * p.c_in * 4) + align256((size_t)p.c_out * p.c_in * p.kh * p.kw * 6);
  if (!tc_eligible(dtype, p)) return 0;
  const size_t nhwc = align256((size_t)p.batch * p.in_h * p.in_w * p.c_in * 2);
  const size_t w = align256((size_t)p.c_out * p.c_in * p.kh * p.kw * 2);
  return nhwc + w;
}

int deform_conv2d_tc_try(const void* input, const void* weight, const void* offset, const void* mask, const void* bias,
                         void* out, int dtype, const DcnParams& p, void* workspace, size_t workspace_bytes, cudaStream_t st,
                         const DcnHints& hints) {
  if (tc3_eligible(dtype, p)) return launch_tc3(input, weight, offset, mask, bias, out, p, workspace, workspace_bytes, st, hints);
  if (!tc_eligible(dtype, p)) return 0;
  if (dtype == VB200_BF16)
    return launch_tc<__nv_bfloat16>(input, weight, offset, mask, bias, out, p, workspace, workspace_bytes, st, hints);
  return launch_tc<__half>(input, weight, offset, mask, bias, out, p, workspace, workspace_bytes, st, hints);
}

// Packed-weight image for the tensor-core path of this shape (0: the shape does not take that path).
size_t deform_conv2d_tc_packed_bytes(int dtype, const DcnParams& p) {
  if (tc3_eligible(dtype, p)) return align256((size_t)p.c_out * p.c_in * p.kh * p.kw * 6);
  if (tc_eligible(dtype, p)) return align256((size_t)p.c_out * p.c_in * p.kh * p.kw * 2);
  return 0;
}
int deform_conv2d_tc_pack(const void* weight, void* packed, int dtype, const DcnParams& p, cudaStream_t st) {
  if (tc3_eligible(dtype, p)) {
    pack_weights3_kernel<<<sm_count() * 4, 256, 0, st>>>((const float*)weight, (__nv_bfloat16*)packed, p.c_out, p.c_in, p.kh * p.kw, tc3_pick_bn(p));
    return check_launch("pack_weights3_kernel");
  }
  if (dtype == VB200_BF16) return pack_tc_weights<__nv_bfloat16>(weight, (__nv_bfloat16*)packed, p, st);
  return pack_tc_weights<__half>(weight, (__half*)packed, p, st);
}

}  // namespace vb200
