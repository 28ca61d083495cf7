// tcgen05 engine for the NeRF MLP (SPARF_ENGINE_TC_3X / TC_1X / TC_3X_W1), sm_100a.
//
// CHAIN KERNELS (tc_mlp_fwd_kernel, tc_mlp_dgrad_kernel): persistent, warp-specialised, one CTA per SM.  A CTA owns
// 128 sample rows at a time (one TMEM lane per row) and pushes them through all tensor-core layers without the
// activations leaving the SM.  Default variant (kTmemA, DESIGN.md 3.1): the A operand of every layer lives in TENSOR
// MEMORY -- TMEM = one 256-column fp32 accumulator | A hi | A lo --
//   warp 0      weight producer : streams pre-packed 16-bit (hi | lo) weight chunks, 16 KB each, from L2 into an
//                                 8..10-stage shared-memory ring with cp.async.bulk + mbarrier complete_tx
//   warp 1      MMA issuer      : an elected lane issues tcgen05.mma M128 x N256 x K16 (A from TMEM, B = two adjacent
//                                 ring stages; the encoder block's A from shared memory), commits to mbarriers
//   warps 2-17  epilogue        : positional encoding (forward); per layer: whole accumulator share -> registers,
//                                 accumulator handed back, then per 64-column block bias/ReLU or mask -> (hi, lo) split
//                                 -> tcgen05.st -> the MMA warp starts the next layer on that K block; density row,
//                                 colour head (128 -> 3) and activations in fp32 on CUDA cores
//   warp 19     image store     : bulk-copies the staged bf16 tape / gradient images from shared memory to HBM
// The forward keeps the older generation for the calls the TMEM kernel does not serve (single-pass engine, bf16
// recompute forward of the backward): operands in shared memory with two N128 issuer warps (warps 1 and 18).
//
// BACKWARD (tc_mlp_backward_tape; tc_mlp_backward re-runs the forward in bf16 "save" mode first):
//   1. the taped forward dumped every layer's A-operand image (bf16 hi | lo) and 64-bit ReLU masks,
//   2. tc_mlp_dgrad_kernel (transposed weights) chains dL/dz_l from the colour head down to layer 0 and dumps each
//      dL/dz_l image,
//   3. tc_mlp_wgrad_kernel computes dW_l = (dL/dz_l)^T x_l: the saved images are consumed AS THEY ARE through MN-major
//      descriptors (reduction over rows), fp32 accumulation in TMEM, one atomic flush per CTA; its reducer warps sum
//      the gradient blocks over rows (bias gradients),
//   4. small CUDA-core kernels finish the density row, the 128 -> 3 head and the view-direction part,
//   5. tc_mlp_encgrad_kernel (pose optimisation): dL/d(encoding) on tensor cores, encoding backward + per-ray sums.
//
// PRECISION: x*W = x_hi*W_hi + x_lo*W_hi + x_hi*W_lo with 16-bit operand halves and fp32 accumulation
// (SURVEY.md hard part 1).  Forward halves are fp16 (2^-22 relative: fp32-like), backward halves are bf16
// (2^-17, full exponent range for tiny gradients).  TC_1X keeps only the first term.  The first layer's
// inputs (x = o + t d, sin/cos of x * 2^j pi) use the reference's exact fp32 op sequence before the split.
//
// Reference: NeRF.forward_samples / forward / compute_raw_density (source/models/frequency_nerf.py:149-281).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "mlp_simt.cuh"
#include "mlp_tc.cuh"
#include "tc_common.cuh"

namespace sparf {
using namespace tc;

namespace {

constexpr int kW = 256;          // trunk width
constexpr int kHW = 128;         // head width
constexpr int kL = 10;           // L_xyz
constexpr int kLv = 4;           // L_view
constexpr int kEv = 27;
constexpr int kNumLayers = 9;    // forward tensor-core layers: trunk 0..7 + head 0
constexpr int kNumBwdLayers = 8; // backward tensor-core layers
constexpr int kTileM = 128;
constexpr int kStages = 3;         // weight-ring stages of the shared-memory-operand forward kernel
constexpr int kMaxStages = 10;
constexpr int kChunkBytes = 16384;  // one [128 x 64] 16-bit operand block
constexpr int kEpiWarps = 16;       // 4 TMEM lane quadrants x 4 column quarters of every 64-column block
constexpr int kEpiCols = 16;        // columns per epilogue warp and block
constexpr int kIssuers = 2;                     // MMA-issuing warps of a stand-alone CTA: warp 1 owns accumulator columns
                                               // 0..127 (N half 0), the warp after the epilogue warps owns N half 1.
                                               // One warp alone spends ~800 clk of dependent uniform-datapath work per
                                               // 16 KB weight chunk, more than the chunk's 256..512 clk of tensor work.
constexpr int kThreads = 64 + 32 * kEpiWarps + 32 * (kIssuers - 1) + 32;  // 640; the last warp (dgrad) streams the
                                               // gradient images from shared memory to HBM with bulk copies
constexpr int kChunksPerTile = 128;     // forward weight chunks per tile
constexpr int kBwdChunksPerTile = 120;  // backward (transposed) weight chunks per tile

// forward: K blocks of a layer: enc first (available early), then the 4 activation blocks
__host__ __device__ constexpr int layer_nkb(int l) { return l == 0 ? 1 : (l == 4 ? 5 : 4); }
__host__ __device__ constexpr int layer_nh(int l) { return l == 8 ? 1 : 2; }     // N / 128
__host__ __device__ constexpr bool kb_is_enc(int l, int kbi) { return l == 0 || (l == 4 && kbi == 0); }
__host__ __device__ constexpr int kb_act_index(int l, int kbi) { return l == 4 ? kbi - 1 : kbi; }
// backward layer bl: 0: g_hid(128) -> g_featpre ; 1: g_featpre -> G6 ; 2..7: G_l -> G_{l-1}, l = 8 - bl
__host__ __device__ constexpr int bwd_nkb(int bl) { return bl == 0 ? 2 : 4; }

// ---- shared memory map of the chain kernels (offsets from a 1024-aligned base)
constexpr int kOffAct = 0;                               // 8 blocks: hi kb0..3, lo kb0..3
constexpr int kOffEnc = kOffAct + 8 * kChunkBytes;       // 2 blocks: hi, lo
constexpr int kOffRing = kOffEnc + 2 * kChunkBytes;      // kStages blocks
constexpr int kOffBias = kOffRing + kStages * kChunkBytes;   // 8 x 256 floats (trunk biases; layer 7: rows 1..256)
constexpr int kOffW7r0 = kOffBias + 8 * 256 * 4;         // 256 floats: density row of the last trunk layer
constexpr int kOffW9 = kOffW7r0 + 256 * 4;               // 3 x 128 floats
constexpr int kOffMisc = kOffW9 + 3 * 128 * 4;           // b7[0], b9[0..2], c2f weights [16]
constexpr int kOffPart = kOffMisc + 32 * 4;              // 3 x 128 x 4 floats: partial dots of column quarters 1..3
constexpr int kOffBar = kOffPart + 3 * 128 * 4 * 4;      // mbarriers
constexpr int kMaxSlots = 8;                              // image staging slots (g_ready / s_free barrier pairs)
constexpr int kNumBars = 2 * kMaxStages + 5 + 4 + 2 * kMaxSlots;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16;
static_assert(kSmemBytes + 1024 <= 232448, "shared memory budget exceeded");

// ---- saved operand images (HBM): tensor t, tile, 64-column block, part (hi | lo): 16 KB each
enum { T_ENC = 0, T_H0 = 1, T_FEAT = 8, T_HID = 9, T_GHID = 10, T_G7F = 11, T_G6 = 12, T_G0 = 18, T_COUNT = 19 };
__host__ __device__ constexpr int tensor_nblk(int t) { return t == T_ENC ? 1 : ((t == T_HID || t == T_GHID) ? 2 : 4); }
__host__ __device__ constexpr int t_g(int l) { return T_G6 + (6 - l); }   // image of dL/dz_l, l = 0..6
// ReLU masks of the forward activations (what the dgrad chain needs of them): layer 0..6 = h0..h6, 7 = feat, 8 = hid;
// per (tile, layer, row): 4 x 64 bits, one word per 16-column quarter cq, bit 16 * block + i = column 64 * block + 16 * cq + i
constexpr int kMaskLayers = 9;
constexpr size_t kMaskTileBytes = (size_t)kMaskLayers * 128 * 32;
struct Images {
  uint8_t* ptr[T_COUNT];   // forward tensors (t < T_GHID) may live in a caller-held tape, gradients in the workspace
  uint8_t* mask;           // forward side
  __host__ __device__ uint8_t* at(int t, int tile, int blk, int part) const {
    return ptr[t] + ((((size_t)tile * tensor_nblk(t)) + blk) * 2 + part) * kChunkBytes;
  }
  __host__ __device__ uint2* mask_at(int tile, int layer, int row, int cq) const {
    return reinterpret_cast<uint2*>(mask + (((size_t)tile * kMaskLayers + layer) * 128 + row) * 32 + cq * 8);
  }
};

struct FwdParams {
  const uint8_t* packed;   // kChunksPerTile chunks of 16 KB
  const float* raybias;    // [R,128]: b8 + W8[:,256:283] . dir_enc(ray)
  const float* origins;
  const float* dirs;
  const float* t;
  const float* noise;
  float* sigma;
  float* rgb;
  const float* bias[8];
  const float* w7;         // last trunk layer weight [257,256]
  const float* w9;         // [3,128]
  const float* b9;
  C2F c2f;
  long long M;             // rows of this launch
  int S;
  int num_tiles;
  int passes;              // 3 (compensated) or 1
  int save;                // dump A-operand images: 0 no, 1 (hi, lo) halves, 2 hi halves only (SPARF_ENGINE_TC_3X_W1)
  Images img;
};

struct BwdParams {
  const uint8_t* packed;   // kBwdChunksPerTile transposed chunks
  const float* d_sigma;    // [M]
  const float* d_rgb;      // [M,3]
  const float* sigma;      // recomputed forward outputs
  const float* rgb;
  float* g_raw;            // [M]   dL/d raw density
  float* g_pre;            // [M,4] dL/d colour pre-activation
  const float* w7;         // [257,256] (row 0 = density row)
  const float* w9;         // [3,128]
  long long M;
  int num_tiles;
  int hi_only;             // 1 (SPARF_ENGINE_TC_3X_W1): gradient images read by the weight-gradient kernel only keep their hi half
  Images img;
};

// reference column of internal encoder column ic (frequency_nerf.py:65-68 layout), -1 = zero pad
__host__ __device__ inline int enc_ref_col(int ic) {
  if (ic < 3) return ic;
  if (ic == 3) return -1;
  int p = (ic - 4) >> 1, is_cos = (ic - 4) & 1;
  int c = p / kL, j = p % kL;
  return 3 + c * 2 * kL + is_cos * kL + j;
}

// ------------------------------------------------------------------------------------------------
// weight packing: fp32 nn.Linear tensors -> 16-bit (hi | lo) SW128 operand blocks in stream order
//   forward : for l: for kb: for nh: for part: chunk [128 (n = out) x 64 (k = in)]           = W[n][k]
//   backward: for bl: for kb: for nh: for part: chunk [128 (n = in)  x 64 (k = out)]         = W[k][n]
// ------------------------------------------------------------------------------------------------
struct PackParams {
  int order;               // 0: chunks ordered (K block, N half, part); 1: (K block, part, N half) = N-256 pairing
  const float* w[9];   // trunk 0..7, head 0
  uint8_t* packed;
};

template <bool kF16>
__global__ void pack_weights_kernel(PackParams pp) {
  int chunk = blockIdx.x;
  int l = 0, base = 0;
  for (;; ++l) {
    int n = layer_nkb(l) * layer_nh(l) * 2;
    if (chunk < base + n) break;
    base += n;
  }
  int rel = chunk - base;
  int part = rel & 1, nh = (rel >> 1) % layer_nh(l), kbi = (rel >> 1) / layer_nh(l);
  if (pp.order == 1 && layer_nh(l) == 2) { nh = rel & 1; part = (rel >> 1) & 1; kbi = rel >> 2; }
  const bool enc = kb_is_enc(l, kbi);
  const int ldw = l == 0 ? 63 : (l == 4 ? 319 : (l == 8 ? 283 : 256));
  const float* W = pp.w[l];
  uint8_t* dst = pp.packed + (size_t)chunk * kChunkBytes;
  // one thread = 8 consecutive K elements of one output row = one 16-byte store into the swizzled image
  for (int e = threadIdx.x; e < 128 * 8; e += blockDim.x) {
    const int n = e >> 3, k0 = (e & 7) * 8;
    const int row = (l == 7 ? 1 : 0) + nh * 128 + n;
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = k0 + 2 * i + h;
        int col;
        if (enc) {
          const int rc = enc_ref_col(k);
          col = rc < 0 ? -1 : (l == 0 ? 0 : kW) + rc;
        } else {
          col = kb_act_index(l, kbi) * 64 + k;
        }
        v[h] = col < 0 ? 0.f : __ldg(W + (size_t)row * ldw + col);
      }
      w[i] = (uint32_t)split1<kF16>(v[0], part) | ((uint32_t)split1<kF16>(v[1], part) << 16);
    }
    *reinterpret_cast<uint4*>(dst + sw128_offset(n, k0)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__global__ void pack_weights_bwd_kernel(PackParams pp) {
  int chunk = blockIdx.x;
  int bl = 0, base = 0;
  for (;; ++bl) {
    int n = bwd_nkb(bl) * 2 * 2;
    if (chunk < base + n) break;
    base += n;
  }
  int rel = chunk - base;
  int nh = rel & 1, part = (rel >> 1) & 1, kbi = rel >> 2;   // (K block, part, N half): the two N halves of a part are
                                                             // adjacent, so one N = 256 MMA can span them
  // source layer and its row offset / leading dimension
  const int l = bl == 0 ? 8 : (bl == 1 ? 7 : 8 - bl);
  const int ldw = l == 4 ? 319 : (l == 8 ? 283 : 256);
  const int rowoff = l == 7 ? 1 : 0;
  const float* W = pp.w[l];
  uint8_t* dst = pp.packed + (size_t)chunk * kChunkBytes;
  // thread = (8 K elements, one row n), n fastest across the threads: the transposed reads W[out][in = n] coalesce
  for (int e = threadIdx.x; e < 128 * 8; e += blockDim.x) {
    const int n = e & 127, k0 = (e >> 7) * 8;
    const int in_idx = nh * 128 + n;         // column of W (input feature of the forward layer)
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int out_idx = kbi * 64 + k0 + 2 * i;   // row of W (output feature)
      const float v0 = __ldg(W + (size_t)(rowoff + out_idx) * ldw + in_idx);
      const float v1 = __ldg(W + (size_t)(rowoff + out_idx + 1) * ldw + in_idx);
      w[i] = (uint32_t)split1<false>(v0, part) | ((uint32_t)split1<false>(v1, part) << 16);
    }
    *reinterpret_cast<uint4*>(dst + sw128_offset(n, k0)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// per-ray view-direction encoding (denc [R,32]) and colour-head bias
//   raybias[r][n] = b8[n] + sum_k W8[n][256+k] * denc[r][k]   (fp32, exact path)
__global__ void raybias_kernel(int R, const float* __restrict__ dirs, const float* __restrict__ w8,
                               const float* __restrict__ b8, C2F c2f, float* __restrict__ raybias,
                               float* __restrict__ denc_out) {
  __shared__ float denc[4][32];
  const int rl = threadIdx.x >> 7, n = threadIdx.x & 127;
  const int r = blockIdx.x * 4 + rl;
  if (n < 32) {
    float val = 0.f;
    if (r < R && n < kEv) {
      float dx = dirs[r * 3], dy = dirs[r * 3 + 1], dz = dirs[r * 3 + 2];
      float len = fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
      int c = n < 3 ? n : (n - 3) / (2 * kLv);
      float u = __fdiv_rn(c == 0 ? dx : (c == 1 ? dy : dz), len);
      if (n < 3) {
        val = u;
      } else {
        int rem = (n - 3) - c * 2 * kLv;
        int is_cos = rem >= kLv;
        int j = rem - is_cos * kLv;
        float arg = mul_rn(u, band_freq(j));
        val = mul_rn(is_cos ? cosf(arg) : sinf(arg), band_weight(c2f, kLv, j));
      }
    }
    denc[rl][n] = val;
    if (r < R && denc_out) denc_out[(size_t)r * 32 + n] = val;
  }
  __syncthreads();
  if (r >= R) return;
  float acc = b8[n];
  const float* wrow = w8 + (size_t)n * (kW + kEv) + kW;
#pragma unroll
  for (int k = 0; k < kEv; ++k) acc = fmaf(wrow[k], denc[rl][k], acc);
  raybias[(size_t)r * kHW + n] = acc;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// split 16 fp32 values of one row into hi/lo words and store them as columns [col0, col0+16) of a
// [128 x 64] SW128 block in shared memory; `save_image` writes the same columns of its HBM image (always bf16 halves:
// the gradient kernels work on those).  The HBM stores come last so that the caller's proxy fence + arrive, which
// release the shared-memory copy to the tensor core, do not sit behind them.
struct Split16 { uint32_t hi[8], lo[8]; };
template <bool kF16>
__device__ __forceinline__ void split16(const float (&f)[16], Split16& o) {
#pragma unroll
  for (int i = 0; i < 8; ++i) split2<kF16>(f[2 * i], f[2 * i + 1], o.hi[i], o.lo[i]);
}
// same into an HBM image: this thread's 16 columns are one aligned 32-byte sector of the row in each block (the
// swizzle only permutes its two 16-byte chunks), written with one 256-bit store per block
__device__ __forceinline__ void st_global_256(uint8_t* p, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                              uint32_t b1, uint32_t b2, uint32_t b3) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"l"(p), "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(b2), "r"(b3)
               : "memory");
}
// bf16 hi words only (= the hi words of split16<false>): the single-pass weight-gradient engine's tape
__device__ __forceinline__ void hi16_bf16(const float (&f)[16], uint32_t (&hi)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    hi[i] = *reinterpret_cast<uint32_t*>(&h);
  }
}
__device__ __forceinline__ void store16_image(const Split16& v, int row, int col0, uint8_t* g_hi, uint8_t* g_lo, bool with_lo = true) {
  const uint32_t off = sw128_offset(row, col0) & ~31u;
  if (row & 1) {   // odd rows: the swizzle swaps the two chunks of the sector
    st_global_256(g_hi + off, v.hi[4], v.hi[5], v.hi[6], v.hi[7], v.hi[0], v.hi[1], v.hi[2], v.hi[3]);
    if (with_lo) st_global_256(g_lo + off, v.lo[4], v.lo[5], v.lo[6], v.lo[7], v.lo[0], v.lo[1], v.lo[2], v.lo[3]);
  } else {
    st_global_256(g_hi + off, v.hi[0], v.hi[1], v.hi[2], v.hi[3], v.hi[4], v.hi[5], v.hi[6], v.hi[7]);
    if (with_lo) st_global_256(g_lo + off, v.lo[0], v.lo[1], v.lo[2], v.lo[3], v.lo[4], v.lo[5], v.lo[6], v.lo[7]);
  }
}
__device__ __forceinline__ void store16_part(const uint32_t (&w)[8], int row, int col0, uint8_t* blk) {
#pragma unroll
  for (int c = 0; c < 2; ++c)
    *reinterpret_cast<uint4*>(blk + sw128_offset(row, col0 + c * 8)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}
__device__ __forceinline__ void store16(const Split16& v, int row, int col0, uint8_t* b_hi, uint8_t* b_lo) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const uint32_t off = sw128_offset(row, col0 + c * 8);
    *reinterpret_cast<uint4*>(b_hi + off) = make_uint4(v.hi[4 * c], v.hi[4 * c + 1], v.hi[4 * c + 2], v.hi[4 * c + 3]);
    *reinterpret_cast<uint4*>(b_lo + off) = make_uint4(v.lo[4 * c], v.lo[4 * c + 1], v.lo[4 * c + 2], v.lo[4 * c + 3]);
  }
}

// ------------------------------------------------------------------------------------------------
// shared pieces of the chain kernels
// ------------------------------------------------------------------------------------------------
// wait-time accounting of the warp roles (only with -DSPARF_TC_TRACE; see tools/trace_chain.py)
struct Trace { long long w[4]; long long t0; int n; };
#ifdef SPARF_TC_TRACE
__device__ long long g_tc_trace[148 * 6 * 8];
__device__ long long g_tc_events[512 * 8];   // CTA 0, first 512 weight chunks: producer / issuer timestamps
__device__ __forceinline__ void trace_begin(Trace& tr) { tr.w[0] = tr.w[1] = tr.w[2] = tr.w[3] = 0; tr.n = 0; tr.t0 = clock64(); }
__device__ __forceinline__ void trace_event(long long g, int k) {
#ifdef SPARF_TC_TRACE_EVENTS
  if (blockIdx.x == 0 && g < 512) g_tc_events[g * 8 + k] = clock64();
#endif
}
__device__ __forceinline__ void twait(Trace& tr, int cat, uint64_t* bar, uint32_t ph) {
  long long a = clock64(); mbar_wait(bar, ph); tr.w[cat] += clock64() - a;
}
__device__ __forceinline__ long long trace_tic() { return clock64(); }
__device__ __forceinline__ void trace_toc(Trace& tr, int cat, long long t0) { tr.w[cat] += clock64() - t0; }
__device__ __forceinline__ void trace_end(const Trace& tr, int role) {
  if (blockIdx.x < 148) {
    long long* o = g_tc_trace + ((size_t)blockIdx.x * 6 + role) * 8;
    o[0] = tr.w[0]; o[1] = tr.w[1]; o[2] = tr.w[2]; o[3] = tr.w[3]; o[4] = clock64() - tr.t0;
  }
}
#else
__device__ __forceinline__ void trace_begin(Trace&) {}
__device__ __forceinline__ void trace_event(long long, int) {}
__device__ __forceinline__ void twait(Trace&, int, uint64_t* bar, uint32_t ph) { mbar_wait(bar, ph); }
__device__ __forceinline__ void trace_end(const Trace&, int) {}
__device__ __forceinline__ long long trace_tic() { return 0; }
__device__ __forceinline__ void trace_toc(Trace&, int, long long) {}
#endif

struct ChainSmem {
  uint8_t* base;
  uint8_t* ring;           // nstages x 16 KB weight ring
  int nstages;
  uint64_t *w_full, *w_empty, *a_ready, *d_full, *d_empty;
  uint64_t *g_ready, *s_free;   // dgrad: block j holds a finished gradient image / has been streamed out
  uint32_t* tmem_slot;
};

__device__ __forceinline__ ChainSmem chain_carve(uint8_t* smem, int ring_off, int nstages, int bar_off = kOffBar) {
  ChainSmem s;
  s.base = smem;
  s.ring = smem + ring_off;
  s.nstages = nstages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + bar_off);
  s.w_full = bars;
  s.w_empty = bars + kMaxStages;
  s.a_ready = bars + 2 * kMaxStages;
  s.d_full = s.a_ready + 5;
  s.d_empty = s.d_full + 2;
  s.g_ready = s.d_empty + 2;
  s.s_free = s.g_ready + kMaxSlots;
  s.tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);
  return s;
}

__device__ __forceinline__ void chain_init_barriers(const ChainSmem& s, int n_issuers = kIssuers) {
  // w_empty: the owning issuer's MMA commit + (two-issuer kernels) the other issuer's "seen it": every waiter of a phase
  // must gate the slot's reuse, or the ring can lap a slow waiter and its parity wait aliases
  for (int i = 0; i < s.nstages; ++i) {
    mbar_init(&s.w_full[i], 1);
    mbar_init(&s.w_empty[i], n_issuers);
  }
  for (int i = 0; i < 5; ++i) mbar_init(&s.a_ready[i], kEpiWarps);
  for (int i = 0; i < kMaxSlots; ++i) { mbar_init(&s.g_ready[i], kEpiWarps); mbar_init(&s.s_free[i], 1); }
  for (int i = 0; i < 2; ++i) { mbar_init(&s.d_full[i], n_issuers); mbar_init(&s.d_empty[i], kEpiWarps); }   // d_full: one commit per issuer warp
  fence_barrier_init();
}

// weight producer (warp 0, uniform control flow, an elected lane issues): streams the per-tile sequence of `nchunks`
// 16 KB chunks through the ring.  (Three producer warps, one per stage, measured no faster: the ring is drained by
// the MMA warps, not starved by the copies.)
__device__ __forceinline__ void chain_producer(const ChainSmem& s, const uint8_t* packed, int my_tiles, int nchunks,
                                               bool skip_lo) {
  Trace tr; trace_begin(tr);
  const int n_eff = skip_lo ? nchunks / 2 : nchunks;
  const long long total = (long long)my_tiles * n_eff;
  for (long long g = 0; g < total; ++g) {
    const int c_eff = (int)(g % n_eff);
    const int c = skip_lo ? 2 * c_eff : c_eff;
    const uint32_t stage = (uint32_t)(g % s.nstages), phase = (uint32_t)((g / s.nstages) & 1);
    twait(tr, 0, &s.w_empty[stage], phase ^ 1);
    if (elect_one()) {
      trace_event(g, 0);
      mbar_arrive_expect_tx(&s.w_full[stage], kChunkBytes);
      bulk_g2s(s.ring + stage * kChunkBytes, packed + (size_t)c * kChunkBytes, kChunkBytes, &s.w_full[stage]);
      trace_event(g, 1);
    }
    __syncwarp();
  }
  if ((threadIdx.x & 31) == 0) trace_end(tr, 0);
}

// Same stream in 32 KB copies over stage pairs (s, s + 1): barriers of the EVEN stage only.  The TMEM-operand kernels
// use it: half the copy issues, expect_tx arms, barrier polls and commits per unit of tensor work (inference forward
// 335 -> 324 us, dgrad 307 -> 302 us against 16 KB copies, profiles/r02_notes.md).
__device__ __forceinline__ void chain_producer_pairs(const ChainSmem& s, const uint8_t* packed, int my_tiles, int nchunks) {
  Trace tr; trace_begin(tr);
  const int npairs = nchunks / 2, nring = s.nstages / 2;
  const long long total = (long long)my_tiles * npairs;
  for (long long g = 0; g < total; ++g) {
    const int c = (int)(g % npairs);
    const uint32_t stage = 2u * (uint32_t)(g % nring), phase = (uint32_t)((g / nring) & 1);
    twait(tr, 0, &s.w_empty[stage], phase ^ 1);
    if (elect_one()) {
      mbar_arrive_expect_tx(&s.w_full[stage], 2 * kChunkBytes);
      bulk_g2s(s.ring + stage * kChunkBytes, packed + (size_t)c * 2 * kChunkBytes, 2 * kChunkBytes, &s.w_full[stage]);
    }
    __syncwarp();
  }
  if ((threadIdx.x & 31) == 0) trace_end(tr, 0);
}

// one (K block, N half): waits for its weight chunks and issues the MMAs of all passes.  Called by the WHOLE issuer
// warp (uniform control flow and operands); one elected lane issues.
__device__ __forceinline__ void chain_issue_block(const ChainSmem& s, uint32_t& stage, uint32_t& phase, uint32_t a_hi,
                                                  uint32_t a_lo, uint32_t d_addr, uint32_t idesc, bool first_kb, int passes,
                                                  bool mine, Trace& tr) {
  const uint32_t ring_addr = smem_u32(s.ring);
  if (!mine) {
    // The other issuer warp's chunks.  They are still waited for: a waiter that skipped a phase of w_full[stage] could
    // later find itself two phases ahead of the barrier, and a parity wait cannot tell "two ahead" from "complete".
    // One combined poll covers the (hi, lo) pair.
    const uint32_t s0 = stage, p0 = phase;
    if (++stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
    if (passes == 1) {
      mbar_wait(&s.w_full[s0], p0);
      if (elect_one()) mbar_arrive(&s.w_empty[s0]);
      __syncwarp();
      return;
    }
    const uint32_t s1 = stage;
    mbar_wait_two(&s.w_full[s0], p0, &s.w_full[s1], phase);
    if (elect_one()) { mbar_arrive(&s.w_empty[s0]); mbar_arrive(&s.w_empty[s1]); }
    __syncwarp();
    if (++stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
    return;
  }
  for (int part = 0; part < (passes == 1 ? 1 : 2); ++part) {
    trace_event(tr.n, 2);
    twait(tr, 2, &s.w_full[stage], phase);
    trace_event(tr.n, 3);
    tc_fence_after();
    // descriptor of K step ks = base descriptor + 2 ks in the 16-byte start-address field (everything lies below
    // 256 KB: no carry), upper word constant: one add per operand instead of the full bit-field assembly
    const uint64_t db0 = make_smem_desc(ring_addr) + (uint64_t)(stage * (kChunkBytes >> 4));
    const uint64_t dah0 = make_smem_desc(a_hi), dal0 = make_smem_desc(a_lo);
    if (elect_one()) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t db = db0 + (uint64_t)(2 * ks);
        const uint32_t acc = (first_kb && part == 0 && ks == 0) ? 0u : 1u;
        umma_ss(d_addr, dah0 + (uint64_t)(2 * ks), db, idesc, acc);
        if (part == 0 && passes != 1) umma_ss(d_addr, dal0 + (uint64_t)(2 * ks), db, idesc, 1u);
      }
      trace_event(tr.n, 4);
      umma_commit(&s.w_empty[stage]);   // frees the ring slot when these MMAs have read it
      trace_event(tr.n, 5);
    }
    __syncwarp();
    ++tr.n;
    if (++stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
  }
}

// N = 256 variant for rings whose chunk order is (K block, part, N half), filled by chain_producer_pairs: the two N
// halves of a part sit in adjacent stages, i.e. form one [256 x 64] K-major operand, and ONE M128 x N256 MMA covers
// them.  Half the instructions and barrier round trips per unit of tensor work (one issuer warp suffices) and
// 96 instead of 128 B/clk of shared-memory operand fetch.
__device__ __forceinline__ void chain_issue_pair256(const ChainSmem& s, uint32_t& stage, uint32_t& phase, uint32_t a_hi,
                                                    uint32_t a_lo, uint32_t d_addr, uint32_t idesc, bool first_kb, Trace& tr) {
  const uint32_t ring_addr = smem_u32(s.ring);
  for (int part = 0; part < 2; ++part) {
    long long t0 = trace_tic();
    mbar_wait(&s.w_full[stage], phase);
    trace_toc(tr, 2, t0);
    tc_fence_after();
    const uint64_t db0 = make_smem_desc(ring_addr) + (uint64_t)(stage * (kChunkBytes >> 4));
    const uint64_t dah0 = make_smem_desc(a_hi), dal0 = make_smem_desc(a_lo);
    if (elect_one()) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t db = db0 + (uint64_t)(2 * ks);
        const uint32_t acc = (first_kb && part == 0 && ks == 0) ? 0u : 1u;
        umma_ss(d_addr, dah0 + (uint64_t)(2 * ks), db, idesc, acc);
        if (part == 0) umma_ss(d_addr, dal0 + (uint64_t)(2 * ks), db, idesc, 1u);
      }
      umma_commit(&s.w_empty[stage]);
    }
    __syncwarp();
    stage += 2;
    if (stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
  }
}

// Same with the A operand in tensor memory (columns a_hi_t / a_lo_t of this K block, +8 columns per K16 step): the MMA
// fetches only B from shared memory and the epilogue hands activations over with tcgen05.st instead of swizzled
// st.shared + fence.proxy.async.
__device__ __forceinline__ void chain_issue_pair256_ts(const ChainSmem& s, uint32_t& stage, uint32_t& phase, uint32_t a_hi_t,
                                                       uint32_t a_lo_t, uint32_t d_addr, uint32_t idesc, bool first_kb, Trace& tr) {
  const uint32_t ring_addr = smem_u32(s.ring);
  for (int part = 0; part < 2; ++part) {
    long long t0 = trace_tic();
    mbar_wait(&s.w_full[stage], phase);
    trace_toc(tr, 2, t0);
    tc_fence_after();
    // descriptor of K step ks = descriptor of the stage + 2 ks in its 16-byte start-address field (no carry: the ring
    // lies below 256 KB), upper word constant: one add per MMA instead of the full bit-field assembly
    const uint64_t db0 = make_smem_desc(ring_addr) + (uint64_t)(stage * (kChunkBytes >> 4));
    if (elect_one()) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t db = db0 + (uint64_t)(2 * ks);
        const uint32_t acc = (first_kb && part == 0 && ks == 0) ? 0u : 1u;
        umma_ts(d_addr, a_hi_t + ks * 8, db, idesc, acc);
        if (part == 0) umma_ts(d_addr, a_lo_t + ks * 8, db, idesc, 1u);
      }
      umma_commit(&s.w_empty[stage]);
    }
    __syncwarp();
    stage += 2;
    if (stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
  }
}

// one [128 x 64] weight chunk against an A operand in tensor memory (the N = 128 colour-head layer): its (hi, lo) parts
// arrive together in the stage pair (stage, stage + 1)
__device__ __forceinline__ void chain_issue_single_ts(const ChainSmem& s, uint32_t& stage, uint32_t& phase, uint32_t a_hi_t,
                                                      uint32_t a_lo_t, uint32_t d_addr, uint32_t idesc, bool first_kb, Trace& tr) {
  const uint32_t ring_addr = smem_u32(s.ring);
  twait(tr, 2, &s.w_full[stage], phase);
  tc_fence_after();
  const uint64_t db0 = make_smem_desc(ring_addr) + (uint64_t)(stage * (kChunkBytes >> 4));
  if (elect_one()) {
#pragma unroll
    for (int part = 0; part < 2; ++part) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t db = db0 + (uint64_t)(part * (kChunkBytes >> 4) + 2 * ks);
        const uint32_t acc = (first_kb && part == 0 && ks == 0) ? 0u : 1u;
        umma_ts(d_addr, a_hi_t + ks * 8, db, idesc, acc);
        if (part == 0) umma_ts(d_addr, a_lo_t + ks * 8, db, idesc, 1u);
      }
    }
    umma_commit(&s.w_empty[stage]);
  }
  __syncwarp();
  stage += 2;
  if (stage == (uint32_t)s.nstages) { stage = 0; phase ^= 1; }
}

// ------------------------------------------------------------------------------------------------
// the fused forward kernel
// ------------------------------------------------------------------------------------------------
// kTmemA (3 passes, fp16 halves): the A operand of every layer except the encoder block lives in tensor memory.
//   TMEM  [0,256) ONE accumulator | [256,384) A hi | [384,512) A lo (32 columns per K block)
//   smem  [0,32K) encoder operand (hi, lo) | taping: [32K,80K) three rotating 16 KB staging slots for the bf16 tape
//         images + an 8-stage weight ring; inference: a 10-stage ring | bias / small weights / barriers as before
// One issuer warp (M128 x N256 MMAs over paired ring stages), the epilogue drains its whole share of the accumulator
// into registers and frees it at once; warp 19 streams the tape images out of the staging slots with bulk copies.
// Image staging (taped forward: kFwdSlots x 16 KB, one (block, part) each; dgrad: kDgSlots x 32 KB, one block's hi | lo).
// The store warp keeps one bulk store in flight: it hands a slot back to the epilogue warps as soon as
// `cp.async.bulk.wait_group.read 0` reports the slot read.  Measured (profiles/r02_notes.md): one store at a time costs
// ~1000 clk per 16 KB copy and the epilogue warps wait 12 % (forward) / 19 % (dgrad) of the kernel for a free slot --
// yet trading ring stages for slots (forward 5 slots + 6 stages, dgrad 3 + 8) or keeping 2-3 stores in flight measured
// SLOWER (taped forward 435 -> 453..461 us, dgrad 291 -> 312..370 us): the weight ring's depth is worth more than the
// slots.  So did copying with ld.shared / st.global instead of bulk copies (taped forward 427 -> 436 us, dgrad 306 ->
// 337 us): the store warp then shares issue slots and the LSU with the epilogue warps.
constexpr int kFwdSlots = 3, kDgSlots = 2;
static_assert(kFwdSlots <= kMaxSlots && kDgSlots <= kMaxSlots, "staging slots");
constexpr int kOffEncT = 0;
constexpr int kOffStgT = 2 * kChunkBytes;
constexpr int kOffRingTSave = kOffStgT + kFwdSlots * kChunkBytes, kStagesTSave = 8;
constexpr int kOffRingTInf = 2 * kChunkBytes, kStagesTInf = 10;
// dgrad: the staging slots, a 10-stage ring (5 [256 x 64] operands), the barriers right after it
constexpr int kOffRingDg = kOffAct + kDgSlots * 2 * kChunkBytes, kStagesDg = 10;
constexpr int kOffBarBwd = kOffRingDg + kStagesDg * kChunkBytes;
static_assert(kStagesTSave % 2 == 0 && kStagesTInf % 2 == 0 && kStagesDg % 2 == 0, "N = 256 MMAs pair adjacent ring stages");
static_assert(kOffRingTSave + kStagesTSave * kChunkBytes <= kOffBias && kOffRingTInf + kStagesTInf * kChunkBytes <= kOffBias,
              "tensor-memory-operand forward: shared-memory map");
static_assert(kOffBarBwd + kNumBars * 8 + 16 <= kSmemBytes, "dgrad shared-memory map exceeds the launch size");

// kHiTape (with kTmemA, p.save == 2): the tape images get their bf16 hi halves only (SPARF_ENGINE_TC_3X_W1)
template <bool kF16, bool kTmemA = false, bool kHiTape = false>
__global__ void __launch_bounds__(kThreads, 1) tc_mlp_fwd_kernel(const FwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* s_bias = reinterpret_cast<float*>(smem + kOffBias);
  float* s_w7r0 = reinterpret_cast<float*>(smem + kOffW7r0);
  float* s_w9 = reinterpret_cast<float*>(smem + kOffW9);
  float* s_misc = reinterpret_cast<float*>(smem + kOffMisc);   // [0]=b7[0], [1..3]=b9, [8..23]=c2f weights
  float* s_part = reinterpret_cast<float*>(smem + kOffPart);   // [cq - 1][row][4]
  const ChainSmem cs = !kTmemA ? chain_carve(smem, kOffRing, kStages)
                                : (p.save ? chain_carve(smem, kOffRingTSave, kStagesTSave) : chain_carve(smem, kOffRingTInf, kStagesTInf));
  uint8_t* const enc_blk = smem + (kTmemA ? kOffEncT : kOffEnc);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- one-time setup
  for (int i = tid; i < 8 * 256; i += kThreads) {
    int l = i >> 8, n = i & 255;
    s_bias[i] = p.bias[l][n + (l == 7 ? 1 : 0)];
  }
  for (int i = tid; i < 256; i += kThreads) s_w7r0[i] = p.w7[i];
  for (int i = tid; i < 3 * 128; i += kThreads) s_w9[i] = p.w9[i];
  if (tid == 0) {
    s_misc[0] = p.bias[7][0];
    s_misc[1] = p.b9[0]; s_misc[2] = p.b9[1]; s_misc[3] = p.b9[2];
  }
  if (tid < 16) s_misc[8 + tid] = tid < kL ? band_weight(p.c2f, kL, tid) : 0.f;
  if (tid == 32) chain_init_barriers(cs, kTmemA ? 1 : kIssuers);
  if (warp == 1) {
    tmem_alloc(cs.tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *cs.tmem_slot, 0);   // warp-uniform for the compiler

  const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles b, b + grid, ...

  if (warp == 0) {
    if (kTmemA) chain_producer_pairs(cs, p.packed, my_tiles, kChunksPerTile);
    else chain_producer(cs, p.packed, my_tiles, kChunksPerTile, p.passes == 1);
  } else if (warp == 1 || warp == 2 + kEpiWarps) {
    const int issuer = warp == 1 ? 0 : 1;
    // ============================== MMA issuer ==============================
    if (kTmemA) {
      if (issuer == 0) {
        const uint32_t idesc256 = make_idesc(128, 256, kF16 ? 0 : 1), idesc128 = make_idesc(128, 128, kF16 ? 0 : 1);
        const uint32_t enc_addr = smem_u32(enc_blk);
        uint32_t stage = 0, phase = 0;
        uint32_t a_cnt[5] = {0, 0, 0, 0, 0};
        uint32_t d_cnt = 0;
        Trace tr; trace_begin(tr);
        for (int it = 0; it < my_tiles; ++it) {
          for (int l = 0; l < kNumLayers; ++l) {
            twait(tr, 0, &cs.d_empty[0], (d_cnt & 1) ^ 1);          // every epilogue warp has the previous accumulator in registers
            ++d_cnt;
            tc_fence_after();
            const int nkb = layer_nkb(l);
            for (int kbi = 0; kbi < nkb; ++kbi) {
              if (kb_is_enc(l, kbi)) {                              // encoder block: operand in shared memory
                if (l == 0) { twait(tr, 1, &cs.a_ready[4], a_cnt[4] & 1); ++a_cnt[4]; }
                tc_fence_after();
                chain_issue_pair256(cs, stage, phase, enc_addr, enc_addr + kChunkBytes, tmem_base, idesc256, kbi == 0, tr);
              } else {
                const int a = kb_act_index(l, kbi);
                twait(tr, 1, &cs.a_ready[a], a_cnt[a] & 1);
                ++a_cnt[a];
                tc_fence_after();
                const uint32_t a_hi_t = tmem_base + 256u + (uint32_t)(a * 32), a_lo_t = tmem_base + 384u + (uint32_t)(a * 32);
                if (l == 8) chain_issue_single_ts(cs, stage, phase, a_hi_t, a_lo_t, tmem_base, idesc128, kbi == 0, tr);
                else chain_issue_pair256_ts(cs, stage, phase, a_hi_t, a_lo_t, tmem_base, idesc256, kbi == 0, tr);
              }
            }
            if (elect_one()) umma_commit(&cs.d_full[0]);
            __syncwarp();
          }
        }
        if (lane == 0) trace_end(tr, 1);
      }
    } else {
      const uint32_t idesc = make_idesc(128, 128, kF16 ? 0 : 1);
      const uint32_t act_addr = smem_u32(smem + kOffAct), enc_addr = smem_u32(smem + kOffEnc);
      uint32_t stage = 0, phase = 0;
      uint32_t a_cnt[5] = {0, 0, 0, 0, 0};
      uint32_t d_cnt[2] = {0, 0};
      Trace tr; trace_begin(tr);
      for (int it = 0; it < my_tiles; ++it) {
        for (int l = 0; l < kNumLayers; ++l) {
          const int buf = l & 1;
          twait(tr, 0, &cs.d_empty[buf], (d_cnt[buf] & 1) ^ 1);   // epilogue of the previous user of this accumulator
          ++d_cnt[buf];
          tc_fence_after();
          const int nkb = layer_nkb(l), nh_cnt = layer_nh(l);
          for (int kbi = 0; kbi < nkb; ++kbi) {
            uint32_t a_hi, a_lo;
            if (kb_is_enc(l, kbi)) {
              if (l == 0) { twait(tr, 1, &cs.a_ready[4], a_cnt[4] & 1); ++a_cnt[4]; }
              a_hi = enc_addr; a_lo = enc_addr + kChunkBytes;
            } else {
              int a = kb_act_index(l, kbi);
              twait(tr, 1, &cs.a_ready[a], a_cnt[a] & 1);
              ++a_cnt[a];
              a_hi = act_addr + a * kChunkBytes; a_lo = act_addr + (4 + a) * kChunkBytes;
            }
            tc_fence_after();
            for (int nh = 0; nh < nh_cnt; ++nh)
              chain_issue_block(cs, stage, phase, a_hi, a_lo, tmem_base + (uint32_t)(buf * 256 + nh * 128), idesc,
                                kbi == 0, p.passes, nh_cnt == 1 ? issuer == 0 : nh == issuer, tr);
          }
          if (elect_one()) umma_commit(&cs.d_full[buf]);            // this warp's share of layer l's accumulator complete
          __syncwarp();
        }
      }
      if (lane == 0 && issuer == 0) trace_end(tr, 1);
    }
  } else if (kTmemA && warp >= 2 + kEpiWarps) {
    // ============================== tape store warp (warp 19) ==============================
    // stream the bf16 tape images of layers 0..7 out of the rotating staging slots (one 16 KB block each)
    if (p.save) {
      uint8_t* stg = smem + kOffStgT;
      constexpr int nparts = kHiTape ? 1 : 2;
      Trace tr; trace_begin(tr);
      for (int it = 0; it < my_tiles; ++it) {
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        for (int l = 0; l < 8; ++l) {
          const int t_img = l == 7 ? T_FEAT : T_H0 + l;
          for (int jq = 0; jq < 4 * nparts; ++jq) {                // (block j, part)
            const int jp = nparts == 2 ? jq : 2 * jq;
            const uint32_t qs = (uint32_t)nparts * (32u * (uint32_t)it + 4u * (uint32_t)l) + (uint32_t)jq;
            const uint32_t slot = qs % (uint32_t)kFwdSlots, k = qs / (uint32_t)kFwdSlots;
            twait(tr, 0, &cs.g_ready[slot], k & 1);
            long long t0 = trace_tic();
            if (elect_one()) {
              bulk_s2g(p.img.at(t_img, tile, jp >> 1, jp & 1), stg + (size_t)slot * kChunkBytes, kChunkBytes);
              bulk_commit_group();
              bulk_wait_read_all();
              mbar_arrive(&cs.s_free[slot]);
            }
            __syncwarp();
            trace_toc(tr, 1, t0);
          }
        }
      }
      if (elect_one()) bulk_wait_all();
      __syncwarp();
      if (lane == 0) trace_end(tr, 4);
    }
  } else if (warp < 2 + kEpiWarps) {
    // ============================== epilogue warps ==============================
    const int e = warp - 2;
    const int q = warp & 3;           // TMEM lane quadrant this warp may access
    const int cq = e >> 2;            // which 16-column quarter of every 64-column block
    const int row = q * 32 + lane;
    const uint32_t t_lane = (uint32_t)(q * 32) << 16;
    uint32_t d_cnt[2] = {0, 0};
    uint8_t* act_hi = smem + kOffAct;
    uint8_t* act_lo = smem + kOffAct + 4 * kChunkBytes;
    const float* wts = s_misc + 8;
    Trace tr; trace_begin(tr);

    for (int it = 0; it < my_tiles; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const long long m = (long long)tile * kTileM + row;
      const bool valid = m < p.M;
      const long long ray = valid ? m / p.S : 0;
      const bool save = p.save != 0;
      constexpr int nparts = kHiTape ? 1 : 2;      // halves of the tape images that are written

      // ---------------- positional encoding -> A_enc (internal column order: x y z 0 | (sin,cos) pairs)
      {
        long long tenc = trace_tic();
        float x[3] = {0.f, 0.f, 0.f};
        if (valid) {
          float tv = p.t[m];
#pragma unroll
          for (int c = 0; c < 3; ++c) x[c] = add_rn(p.origins[ray * 3 + c], mul_rn(p.dirs[ray * 3 + c], tv));
        }
        float vals[16];
        if (cq == 0) { vals[0] = x[0]; vals[1] = x[1]; vals[2] = x[2]; vals[3] = 0.f; }
        const int p0 = cq == 0 ? 0 : 8 * cq - 2, np = cq == 0 ? 6 : 8, v0 = cq == 0 ? 4 : 0;   // 6 + 8 + 8 + 8 pairs
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (i < np) {
            int pr = p0 + i;
            int c = pr / kL, j = pr - c * kL;
            float arg = mul_rn(c == 0 ? x[0] : (c == 1 ? x[1] : x[2]), band_freq(j));
            float sn, cs_;
            sincosf(arg, &sn, &cs_);
            float w = wts[j];
            vals[v0 + 2 * i] = mul_rn(sn, w);
            vals[v0 + 2 * i + 1] = mul_rn(cs_, w);
          }
        }
        Split16 sp;
        split16<kF16>(vals, sp);
        store16(sp, row, cq * kEpiCols, enc_blk, enc_blk + kChunkBytes);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&cs.a_ready[4]);
        if (save) {
          if (kF16) split16<false>(vals, sp);
          // (both halves whatever the tape mode: the ray-gradient kernel rebuilds sin / cos from this image)
          store16_image(sp, row, cq * kEpiCols, p.img.at(T_ENC, tile, 0, 0), p.img.at(T_ENC, tile, 0, 1));
        }
        trace_toc(tr, 3, tenc);
      }

      // ---------------- layers
      for (int l = 0; l < kNumLayers; ++l) {
        const int buf = kTmemA ? 0 : (l & 1);
        twait(tr, 0, &cs.d_full[buf], d_cnt[buf] & 1);
        ++d_cnt[buf];
        tc_fence_after();
        const int nchunk = l == 8 ? 2 : 4;
        float dot0 = 0.f, dot1 = 0.f, dot2 = 0.f;   // density row (l == 6) or rgb rows (l == 8)
        uint32_t mbits[2] = {0u, 0u};               // ReLU mask of this thread's 16 columns in each block
        uint32_t vn[16];                            // accumulator columns of the NEXT block, loaded one block ahead
        uint32_t va[kTmemA ? 4 : 1][16];            // kTmemA: this thread's whole share of the accumulator
        if (kTmemA) {
          long long tld = trace_tic();
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < nchunk) tmem_ld16(tmem_base + t_lane + (uint32_t)(j * 64 + cq * kEpiCols), va[j]);
          tmem_ld_wait();
          trace_toc(tr, 2, tld);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&cs.d_empty[0]);   // the (single) accumulator is free for the next layer's MMAs
        } else {
          tmem_ld16(tmem_base + t_lane + (uint32_t)(buf * 256 + cq * kEpiCols), vn);
        }
        if (kTmemA && l < 8) {
          // ---- phase 1 (critical path): bias + ReLU -> fp16 (hi, lo) -> tensor memory, block by block; the MMA warp
          // starts layer l + 1 on K block j as soon as block j is in.  The activations stay in va[] for phase 2.
          const float* bl_ = s_bias + l * 256 + cq * kEpiCols;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float f[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              f[i] = fmaxf(__uint_as_float(va[j][i]) + bl_[j * 64 + i], 0.f);
              va[j][i] = __float_as_uint(f[i]);
            }
            Split16 sp;
            split16<kF16>(f, sp);
            tmem_st8(tmem_base + t_lane + 256u + (uint32_t)(j * 32 + cq * 8), sp.hi);
            tmem_st8(tmem_base + t_lane + 384u + (uint32_t)(j * 32 + cq * 8), sp.lo);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&cs.a_ready[j]);
          }
          // ---- phase 2 (overlaps the next layer's MMAs): density row, ReLU masks, bf16 tape through the staging slots
          if (l == 6 || save) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int col0 = j * 64 + cq * kEpiCols;
              float f[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(va[j][i]);
              if (l == 6) {
#pragma unroll
                for (int i = 0; i < 16; ++i) dot0 = fmaf(f[i], s_w7r0[col0 + i], dot0);
              }
              if (save) {
                uint32_t m16 = 0;
#pragma unroll
                for (int i = 0; i < 16; ++i) m16 |= (f[i] > 0.f ? 1u : 0u) << i;
                mbits[j >> 1] |= m16 << (16 * (j & 1));
                Split16 sp;
                if (nparts == 2) split16<false>(f, sp); else hi16_bf16(f, sp.hi);
                uint8_t* stg = smem + kOffStgT;
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                  if (part >= nparts) break;
                  const uint32_t qs = (uint32_t)nparts * (32u * (uint32_t)it + 4u * (uint32_t)l + (uint32_t)j) + (uint32_t)part;
                  const uint32_t slot = qs % (uint32_t)kFwdSlots, k = qs / (uint32_t)kFwdSlots;
                  if (k > 0) twait(tr, 1, &cs.s_free[slot], (k - 1) & 1);
                  store16_part(part == 0 ? sp.hi : sp.lo, row, cq * kEpiCols, stg + (size_t)slot * kChunkBytes);
                  fence_proxy_async_smem();
                  __syncwarp();
                  if (lane == 0) mbar_arrive(&cs.g_ready[slot]);
                }
              }
            }
          }
        } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j >= nchunk) break;
          uint32_t v[16];
          const int col0 = j * 64 + cq * kEpiCols;
          if (kTmemA) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = va[j][i];
          } else {
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = vn[i];
            if (j + 1 < nchunk) tmem_ld16(tmem_base + t_lane + (uint32_t)(buf * 256 + col0 + 64), vn);
          }
          float f[16];
          if (l < 8) {
            const float* b = s_bias + l * 256 + col0;
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] = fmaxf(__uint_as_float(v[i]) + b[i], 0.f);
          } else {
            const float* b = p.raybias + (size_t)ray * kHW + col0;
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              float4 bb = *reinterpret_cast<const float4*>(b + i);
              f[i] = fmaxf(__uint_as_float(v[i]) + bb.x, 0.f);
              f[i + 1] = fmaxf(__uint_as_float(v[i + 1]) + bb.y, 0.f);
              f[i + 2] = fmaxf(__uint_as_float(v[i + 2]) + bb.z, 0.f);
              f[i + 3] = fmaxf(__uint_as_float(v[i + 3]) + bb.w, 0.f);
            }
          }
          if (l == 6) {
#pragma unroll
            for (int i = 0; i < 16; ++i) dot0 = fmaf(f[i], s_w7r0[col0 + i], dot0);
          }
          if (save) {
            uint32_t m16 = 0;
#pragma unroll
            for (int i = 0; i < 16; ++i) m16 |= (f[i] > 0.f ? 1u : 0u) << i;
            mbits[j >> 1] |= m16 << (16 * (j & 1));
          }
          Split16 sp;
          if (l == 8) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              dot0 = fmaf(f[i], s_w9[col0 + i], dot0);
              dot1 = fmaf(f[i], s_w9[128 + col0 + i], dot1);
              dot2 = fmaf(f[i], s_w9[256 + col0 + i], dot2);
            }
            if (save) {   // hid image for the 128->3 head's weight gradient and its ReLU mask
              split16<false>(f, sp);
              store16_image(sp, row, cq * kEpiCols, p.img.at(T_HID, tile, j, 0), p.img.at(T_HID, tile, j, 1), nparts == 2);
            }
          } else {
            split16<kF16>(f, sp);
            store16(sp, row, cq * kEpiCols, act_hi + (size_t)j * kChunkBytes, act_lo + (size_t)j * kChunkBytes);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&cs.a_ready[j]);
            if (save) {
              const int tsave = l == 7 ? T_FEAT : T_H0 + l;
              if (kF16) split16<false>(f, sp);
              store16_image(sp, row, cq * kEpiCols, p.img.at(tsave, tile, j, 0), p.img.at(tsave, tile, j, 1), nparts == 2);
            }
          }
        }
        }   // (shared-memory-operand kernels and the colour-head layer)
        // accumulator drained: hand it back to the MMA warp (kTmemA did so right after loading it)
        if (!kTmemA) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&cs.d_empty[buf]);
        }
        if (save) *p.img.mask_at(tile, l, row, cq) = make_uint2(mbits[0], mbits[1]);

        if (l == 6 || l == 8) {
          // combine the four column quarters of each row (warps q, q+4, q+8, q+12) through shared memory
          if (cq != 0) {
            float* pr = s_part + ((size_t)(cq - 1) * 128 + row) * 4;
            pr[0] = dot0; pr[1] = dot1; pr[2] = dot2;
          }
          named_bar_sync(1, kEpiWarps * 32);
          if (cq == 0 && valid) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              const float* o = s_part + ((size_t)k * 128 + row) * 4;
              dot0 += o[0]; dot1 += o[1]; dot2 += o[2];
            }
            if (l == 6) {
              float raw = dot0 + s_misc[0];
              float z = p.noise ? add_rn(raw, p.noise[m]) : raw;
              p.sigma[m] = softplus_f(z);
            } else {
              p.rgb[m * 3 + 0] = sigmoid_f(dot0 + s_misc[1]);
              p.rgb[m * 3 + 1] = sigmoid_f(dot1 + s_misc[2]);
              p.rgb[m * 3 + 2] = sigmoid_f(dot2 + s_misc[3]);
            }
          }
          named_bar_sync(1, kEpiWarps * 32);
        }
      }
    }
    if (lane == 0 && (e == 0 || e == kEpiWarps - 1)) trace_end(tr, e == 0 ? 2 : 3);
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// the fused input-gradient (dgrad) kernel: dL/dz chain from the colour head to layer 0
// ------------------------------------------------------------------------------------------------
// TMEM = [0,256) ONE accumulator | [256,384) A hi | [384,512) A lo (32 columns per K block).
// The epilogue loads its whole share of the accumulator into registers first and hands the accumulator back at once,
// so a single accumulator still lets layer l+1's MMAs overlap layer l's epilogue.  Shared memory holds no A operand:
// kDgSlots rotating (hi, lo) staging slots for the gradient images' bulk stores, then the weight ring.
__global__ void __launch_bounds__(kThreads, 1) tc_mlp_dgrad_kernel(const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // The density row and the 128 -> 3 colour weights (2.5 KB, read by every thread) come from global memory through L1.
  const float* __restrict__ s_w7r0 = p.w7;
  const float* __restrict__ s_w9 = p.w9;
  const ChainSmem cs = chain_carve(smem, kOffRingDg, kStagesDg, kOffBarBwd);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 32) chain_init_barriers(cs, 1);   // ONE issuer warp (N = 256 MMAs)
  if (warp == 1) {
    tmem_alloc(cs.tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *cs.tmem_slot, 0);
  const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    chain_producer_pairs(cs, p.packed, my_tiles, kBwdChunksPerTile);
  } else if (warp == 1 || warp == 2 + kEpiWarps) {
    if (warp == 1) {   // (warp 18 idles)
      const uint32_t idesc = make_idesc(128, 256, 1);
      uint32_t stage = 0, phase = 0;
      uint32_t a_cnt[4] = {0, 0, 0, 0};
      uint32_t d_cnt = 0;
      Trace tr; trace_begin(tr);
      for (int it = 0; it < my_tiles; ++it) {
        for (int bl = 0; bl < kNumBwdLayers; ++bl) {
          twait(tr, 0, &cs.d_empty[0], (d_cnt & 1) ^ 1);
          ++d_cnt;
          tc_fence_after();
          const int nkb = bwd_nkb(bl);
          for (int kbi = 0; kbi < nkb; ++kbi) {
            twait(tr, 1, &cs.a_ready[kbi], a_cnt[kbi] & 1);
            ++a_cnt[kbi];
            tc_fence_after();
            chain_issue_pair256_ts(cs, stage, phase, tmem_base + 256u + (uint32_t)(kbi * 32),
                                   tmem_base + 384u + (uint32_t)(kbi * 32), tmem_base, idesc, kbi == 0, tr);
          }
          if (elect_one()) umma_commit(&cs.d_full[0]);
          __syncwarp();
        }
      }
      if (lane == 0) trace_end(tr, 1);
    }
  } else if (warp >= 2 + kEpiWarps) {
    // ============================== gradient-image store warp (warp 19) ==============================
    // stream every finished [128 x 64] hi / lo block pair (already in the HBM image layout) out of the staging slots
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      for (int step = 0; step <= kNumBwdLayers; ++step) {          // step 0 = head (blocks 0, 1), step bl + 1 = layer bl
        const int nblk = step == 0 ? 2 : 4;
        const int t_out = step == 0 ? T_GHID : (step == 1 ? T_G7F : t_g(8 - step));
        for (int j = 0; j < nblk; ++j) {
          // q = running index of the (tile, step, block) writes: slot q % kDgSlots, q / kDgSlots its per-slot number
          const uint32_t q = 34u * (uint32_t)it + (step == 0 ? (uint32_t)j : 2u + 4u * (uint32_t)(step - 1) + (uint32_t)j);
          const int slot = (int)(q % (uint32_t)kDgSlots);
          const uint8_t* src = smem + kOffAct + (size_t)slot * 2 * kChunkBytes;
          mbar_wait(&cs.g_ready[slot], (q / (uint32_t)kDgSlots) & 1);
          if (elect_one()) {
            // (hi | lo) of a block are adjacent in the slot AND in the HBM image: one 32 KB bulk store.
            // hi_only (SPARF_ENGINE_TC_3X_W1): images only the single-pass weight-gradient kernel reads keep their hi half
            const bool both = !p.hi_only || t_out == T_GHID || step == kNumBwdLayers || t_out == t_g(4);
            bulk_s2g(p.img.at(t_out, tile, j, 0), src, (both ? 2 : 1) * kChunkBytes);
            bulk_commit_group();
            bulk_wait_read_all();
            mbar_arrive(&cs.s_free[slot]);
          }
          __syncwarp();
        }
      }
    }
    if (elect_one()) bulk_wait_all();
    __syncwarp();
  } else {
    const int e = warp - 2;
    const int q = warp & 3;
    const int cq = e >> 2;
    const int row = q * 32 + lane;
    const uint32_t t_lane = (uint32_t)(q * 32) << 16;
    uint32_t d_cnt = 0;
    Trace tr; trace_begin(tr);

    for (int it = 0; it < my_tiles; ++it) {
      const int tile = (int)blockIdx.x + it * (int)gridDim.x;
      const long long m = (long long)tile * kTileM + row;
      const bool valid = m < p.M;

      // ---------------- head: g_pre = d_rgb * c (1 - c); g_raw = d_sigma * (1 - e^-sigma) [= sigmoid(z)];
      //                  g_hid = (hid > 0) * (g_pre . W9)  -> A blocks 0, 1
      float gp0 = 0.f, gp1 = 0.f, gp2 = 0.f, g_raw = 0.f;
      if (valid) {
        float c0 = p.rgb[m * 3], c1 = p.rgb[m * 3 + 1], c2 = p.rgb[m * 3 + 2];
        gp0 = p.d_rgb[m * 3] * c0 * (1.f - c0);
        gp1 = p.d_rgb[m * 3 + 1] * c1 * (1.f - c1);
        gp2 = p.d_rgb[m * 3 + 2] * c2 * (1.f - c2);
        g_raw = p.d_sigma[m] * (-expm1f(-p.sigma[m]));
        if (cq == 0) {
          p.g_raw[m] = g_raw;
          *reinterpret_cast<float4*>(p.g_pre + m * 4) = make_float4(gp0, gp1, gp2, 0.f);
        }
      }
      // Every gradient block goes to tensor memory (the next layer's A operand) and through a staging slot to the store
      // warp; write number k of a slot waits for the store of write k - 1 to have read it (qs numbered as in the store warp)
      const uint2 hid_mask = *p.img.mask_at(tile, 8, row, cq);
#pragma unroll 1
      for (int j = 0; j < 2; ++j) {
        const int col0 = j * 64 + cq * kEpiCols;
        const uint32_t mask = (hid_mask.x >> (16 * j)) & 0xFFFFu;
        float f[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float g = fmaf(gp2, s_w9[256 + col0 + i], fmaf(gp1, s_w9[128 + col0 + i], gp0 * s_w9[col0 + i]));
          f[i] = ((mask >> i) & 1u) ? g : 0.f;
        }
        Split16 sp;
        split16<false>(f, sp);
        tmem_st8(tmem_base + t_lane + 256u + (uint32_t)(j * 32 + cq * 8), sp.hi);
        tmem_st8(tmem_base + t_lane + 384u + (uint32_t)(j * 32 + cq * 8), sp.lo);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&cs.a_ready[j]);
        const uint32_t qs = 34u * (uint32_t)it + (uint32_t)j, k = qs / (uint32_t)kDgSlots;
        const int slot = (int)(qs % (uint32_t)kDgSlots);
        uint8_t* st_hi = smem + kOffAct + (size_t)slot * 2 * kChunkBytes;
        if (k > 0) mbar_wait(&cs.s_free[slot], (k - 1) & 1);
        store16(sp, row, cq * kEpiCols, st_hi, st_hi + kChunkBytes);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&cs.g_ready[slot]);
      }

      // ---------------- backward layers
      for (int bl = 0; bl < kNumBwdLayers; ++bl) {
        // ReLU mask of the forward activation this gradient flows into: feat (bl 0), h6 (bl 1), ... h0 (bl 7)
        long long tt = trace_tic();
        const uint2 mk = *p.img.mask_at(tile, bl == 0 ? 7 : 7 - bl, row, cq);
        const uint32_t masks[2] = {mk.x, mk.y};
        trace_toc(tr, 1, tt);
        twait(tr, 0, &cs.d_full[0], d_cnt & 1);
        ++d_cnt;
        tc_fence_after();
        uint32_t va[4][16];                         // this thread's whole share of the accumulator
        long long tld = trace_tic();
#pragma unroll
        for (int j = 0; j < 4; ++j) tmem_ld16(tmem_base + t_lane + (uint32_t)(j * 64 + cq * kEpiCols), va[j]);
        tmem_ld_wait();
        trace_toc(tr, 2, tld);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&cs.d_empty[0]);   // the (single) accumulator is free for the next layer's MMAs
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int col0 = j * 64 + cq * kEpiCols;
          float f[16];
          const uint32_t mask = (masks[j >> 1] >> (16 * (j & 1))) & 0xFFFFu;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float g = __uint_as_float(va[j][i]);
            if (bl == 1) g = fmaf(g_raw, s_w7r0[col0 + i], g);   // density row joins the feature gradient
            f[i] = ((mask >> i) & 1u) ? g : 0.f;
          }
          Split16 sp;
          split16<false>(f, sp);
          if (bl != kNumBwdLayers - 1) {   // G0 is only saved, nothing consumes it on-chip
            tmem_st8(tmem_base + t_lane + 256u + (uint32_t)(j * 32 + cq * 8), sp.hi);
            tmem_st8(tmem_base + t_lane + 384u + (uint32_t)(j * 32 + cq * 8), sp.lo);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&cs.a_ready[j]);
          }
          long long tt3 = trace_tic();
          const uint32_t qs = 34u * (uint32_t)it + 2u + 4u * (uint32_t)bl + (uint32_t)j, k = qs / (uint32_t)kDgSlots;
          const int slot = (int)(qs % (uint32_t)kDgSlots);
          uint8_t* st_hi = smem + kOffAct + (size_t)slot * 2 * kChunkBytes;
          if (k > 0) mbar_wait(&cs.s_free[slot], (k - 1) & 1);
          trace_toc(tr, 3, tt3);
          store16(sp, row, cq * kEpiCols, st_hi, st_hi + kChunkBytes);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&cs.g_ready[slot]);
        }
      }
    }
    if (lane == 0 && (e == 0 || e == kEpiWarps - 1)) trace_end(tr, e == 0 ? 2 : 3);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// weight-gradient kernel: dW[m'][n'] += sum_rows G[row][m'] * X[row][n'] over a slab of row tiles
// ------------------------------------------------------------------------------------------------
// 8 bf16 (hi, lo) pairs -> fp32
__device__ __forceinline__ void unpack8(const uint4& h, const uint4& l, float (&x)[8]) {
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    x[2 * i] = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
    x[2 * i + 1] = __uint_as_float(hw[i] & 0xFFFF0000u) + __uint_as_float(lw[i] & 0xFFFF0000u);
  }
}

struct WgradJob {
  int t_g, t_x;          // image tensors: gradient (M' side) and activation (N' side)
  int mblk, nblk;        // 64-column blocks on each side (M' = 64 mblk in {128, 256}; N' = 64 nblk in {64, 256})
  int tile_begin, tile_end;
  float* dW;             // destination [*, ldw]
  int ldw, col0;         // row stride and first column
  int enc_cols;          // 1: N' side is the encoder block (internal column order -> reference columns)
  float* colsum;         // optional: colsum[f] += sum_rows G[row][f]  (the layer's bias gradient), else NULL
  int passes;            // 3: G_hi X_hi + G_lo X_hi + G_hi X_lo;  1 (SPARF_ENGINE_TC_3X_W1): G_hi X_hi, the lo halves are
                         // not read at all (the bias gradients become column sums of G_hi)
};
constexpr int kMaxWgradJobs = 160;
struct WgradJobs { WgradJob j[kMaxWgradJobs]; };   // passed by value (kernel parameter): no host->device copy per step
constexpr int kWgStages = 3;                // three passes: 3 stages of 64 KB; one pass (hi halves only): 6 stages of 32 KB, so
constexpr int kWgMaxStages = 6;             // that the same number of bytes is in flight per SM (the kernel is HBM-latency bound)
constexpr int kWgStageBytes = 16 * 4096;   // (4 G blocks + 4 X blocks) x (hi, lo) x 32 rows x 128 B
constexpr int kWgSmem = kWgStages * kWgStageBytes + 256;

__global__ void __launch_bounds__(192, 1) tc_mlp_wgrad_kernel(const __grid_constant__ WgradJobs jobs, const __grid_constant__ Images img) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgStages * kWgStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kWgMaxStages;
  uint64_t* done = bars + 2 * kWgMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWgMaxStages + 1);
  const WgradJob& job = jobs.j[blockIdx.x];
  const bool one_pass = job.passes == 1;
  // one pass: both sides load their hi halves only (the bias gradients = column sums of G are then sums of G_hi too);
  // stage = [G hi: 4 x 4 KB][X hi: 4 x 4 KB], twice as many stages
  const int g_parts = one_pass ? 1 : 2, x_parts = g_parts;
  const uint32_t nstages = one_pass ? 2u * kWgStages : (uint32_t)kWgStages;
  const uint32_t stage_bytes = one_pass ? (uint32_t)kWgStageBytes / 2u : (uint32_t)kWgStageBytes;
  const uint32_t x_blk0 = one_pass ? 4u : 8u;      // first 4 KB block of the X side within a stage
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncols = job.nblk * 64;                       // N'
  const int mhalves = job.mblk / 2;                      // accumulators of 128 rows
  const uint32_t tmem_cols = (mhalves * ncols <= 64) ? 64 : (mhalves * ncols <= 128 ? 128 : (mhalves * ncols <= 256 ? 256 : 512));

  if (tid == 0) {
    for (int i = 0; i < kWgMaxStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 5); }   // MMA commit + 4 reducer warps
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const int nq = (job.tile_end - job.tile_begin) * 4;    // quarter tiles (32 rows) to stream
  const uint32_t stage_tx = (uint32_t)(job.mblk * g_parts + job.nblk * x_parts) * 4096u;

  if (warp == 0) {
    // producer warp (uniform control flow, an elected lane issues).  A second producer warp for the activation side
    // measured no faster: the kernel is bound by HBM latency / bandwidth, not by the issue rate of the copies.
    uint32_t stage = 0, phase = 0;
    for (int qi = 0; qi < nq; ++qi) {
      const int tile = job.tile_begin + (qi >> 2), qr = qi & 3;
      mbar_wait(&empty[stage], phase ^ 1);
      if (elect_one()) {
        uint8_t* st = smem + stage * stage_bytes;
        // stage layout: [G hi: mblk x 4 KB][G lo][X hi: nblk x 4 KB][X lo], 4 KB = rows [32 qr, 32 qr + 32) of a block
        mbar_arrive_expect_tx(&full[stage], stage_tx);
        for (int part = 0; part < 2; ++part) {
          if (part < g_parts)
            for (int b = 0; b < job.mblk; ++b)
              bulk_g2s(st + (part * 4 + b) * 4096, img.at(job.t_g, tile, b, part) + qr * 4096, 4096, &full[stage]);
          if (part < x_parts)
            for (int b = 0; b < job.nblk; ++b)
              bulk_g2s(st + (x_blk0 + part * 4 + b) * 4096, img.at(job.t_x, tile, b, part) + qr * 4096, 4096, &full[stage]);
        }
      }
      __syncwarp();
      if (++stage == nstages) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc(128, ncols, 1, 1, 1);
    uint32_t stage = 0, phase = 0;
    for (int qi = 0; qi < nq; ++qi) {
      mbar_wait(&full[stage], phase);
      tc_fence_after();
      const uint32_t st = smem_u32(smem + stage * stage_bytes);
      if (elect_one()) {
        for (int mh = 0; mh < mhalves; ++mh) {
          const uint32_t d_addr = tmem_base + (uint32_t)(mh * ncols);
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {   // 32 rows = 2 x K16
            const uint64_t g_hi = make_smem_desc_mn(st + (0 + mh * 2) * 4096 + ks * 2048, 4096);
            const uint64_t g_lo = make_smem_desc_mn(st + (4 + mh * 2) * 4096 + ks * 2048, 4096);
            const uint64_t x_hi = make_smem_desc_mn(st + x_blk0 * 4096 + ks * 2048, 4096);
            const uint64_t x_lo = make_smem_desc_mn(st + 12 * 4096 + ks * 2048, 4096);
            umma_ss(d_addr, g_hi, x_hi, idesc, (qi | ks) != 0);
            if (!one_pass) {
              umma_ss(d_addr, g_lo, x_hi, idesc, 1u);
              umma_ss(d_addr, g_hi, x_lo, idesc, 1u);
            }
          }
        }
        umma_commit(&empty[stage]);
      }
      __syncwarp();
      if (++stage == nstages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else {
    // warps 2..5: while the MMA warp streams, reduce the gradient images over the rows straight from the shared
    // memory stages (bias gradient = column sums of G); at the end flush the accumulator with atomics on dW
    const int q = warp & 3;
    const int rowl = q * 32 + lane;
    {
      // reducer warp w owns gradient block w of every stage: lane = (row group rg, 16-byte chunk c); 8 features x 8 rows
      // per thread and stage with conflict-free 16-byte loads (8 consecutive lanes read one swizzled 128-byte row)
      const int blk = warp - 2, c = lane & 7, rg = lane >> 3;
      const bool has = job.colsum && blk < job.mblk;
      float cs[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) cs[k] = 0.f;
      uint32_t stage = 0, phase = 0;
      for (int qi = 0; qi < nq; ++qi) {
        mbar_wait(&full[stage], phase);
        if (has) {
          const uint8_t* bh = smem + stage * stage_bytes + blk * 4096;
          const uint8_t* bl = bh + 4 * 4096;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t off = (uint32_t)(rg * 8 + i) * 128u + (uint32_t)((c ^ i) << 4);
            float x[8];
            unpack8(*reinterpret_cast<const uint4*>(bh + off),
                    one_pass ? make_uint4(0u, 0u, 0u, 0u) : *reinterpret_cast<const uint4*>(bl + off), x);
#pragma unroll
            for (int k = 0; k < 8; ++k) cs[k] += x[k];
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        if (++stage == nstages) { stage = 0; phase ^= 1; }
      }
      if (has) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float v = cs[k];
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          if (rg == 0) atomicAdd(job.colsum + blk * 64 + c * 8 + k, v);
        }
      }
    }
    mbar_wait(done, 0);
    tc_fence_after();
    for (int mh = 0; mh < mhalves; ++mh) {
      float* drow = job.dW + (size_t)(mh * 128 + rowl) * job.ldw + job.col0;
      for (int c0 = 0; c0 < ncols; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mh * ncols + c0), v);
        tmem_ld_wait();
        if (nq > 0) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            int col = c0 + i;
            if (job.enc_cols) {
              col = enc_ref_col(col);
              if (col < 0) continue;
            }
            atomicAdd(drow + col, __uint_as_float(v[i]));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// CUDA-core helpers on the saved images
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float img_value(const Images& img, int t, long long m, int f) {
  const int tile = (int)(m >> 7), row = (int)(m & 127);
  const uint32_t off = sw128_offset(row, f & 63);
  const uint16_t hi = *reinterpret_cast<const uint16_t*>(img.at(t, tile, f >> 6, 0) + off);
  const uint16_t lo = *reinterpret_cast<const uint16_t*>(img.at(t, tile, f >> 6, 1) + off);
  return __uint_as_float((uint32_t)hi << 16) + __uint_as_float((uint32_t)lo << 16);
}

// One row-reduction over the saved images per launch (bias gradients and the two narrow layers):
//   mode 0:  out[f]            += sum_m img[m][f]                                   (colsum -> bias grads)
//   mode 1/3: out[c*ldo + f]   += sum_m g[m*gs + c] * img[m][f], out_bias[c] += sum_m g[m*gs + c]
// Block = 256 threads = 8 row groups x 32 sixteen-byte chunks (8 features each); a block owns a few row
// tiles, reads them with 16-byte loads along the swizzled rows, reduces in shared memory, one atomic per
// feature per block.
struct ReduceJob {
  int t, nblk, nc;     // image tensor, 64-feature blocks (2 or 4), nc = 0 (colsum), 1 or 3 (narrow outputs)
  const float* g;
  int gs;
  float* out;
  int ldo;
  float* out_bias;
  int parts;           // 2: image = hi + lo halves; 1: hi half only (the lo half was not written: SPARF_ENGINE_TC_3X_W1)
};

template <int NC>   // NC = 0 (column sums) | 1 | 3 narrow outputs: sizes the accumulators (registers -> blocks per SM)
__global__ void __launch_bounds__(256) image_reduce_kernel(const __grid_constant__ ReduceJob job, Images img, long long M,
                                                           int ntiles, int tiles_per_block) {
  __shared__ float red[8][32][25];
  const int tid = threadIdx.x, c16 = tid & 31, rg = tid >> 5;
  const int fb = c16 >> 3, c = c16 & 7;
  const bool active = fb < job.nblk;
  constexpr int nc = NC;
  constexpr int kAcc = NC == 0 ? 8 : NC * 8;
  float acc[kAcc];
#pragma unroll
  for (int i = 0; i < kAcc; ++i) acc[i] = 0.f;
  float accb[3] = {0.f, 0.f, 0.f};
  const int t0 = blockIdx.x * tiles_per_block, t1 = min(ntiles, t0 + tiles_per_block);
  for (int tile = t0; tile < t1; ++tile) {
    const uint8_t* bh = img.at(job.t, tile, active ? fb : 0, 0);
    const uint8_t* bl = img.at(job.t, tile, active ? fb : 0, 1);
    if (!active) continue;
#pragma unroll 1
    for (int r0 = rg; r0 < 128; r0 += 32) {     // 4 rows per pass: 8 independent 16-byte loads in flight per thread
      uint4 vh[4], vl[4];
      float gv[4][3];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int row = r0 + 8 * u;
        const long long m = (long long)tile * 128 + row;
        const uint32_t off = sw128_offset(row, c * 8);
        const bool ok = m < M;
        vh[u] = ok ? __ldg(reinterpret_cast<const uint4*>(bh + off)) : make_uint4(0, 0, 0, 0);
        vl[u] = (ok && job.parts == 2) ? __ldg(reinterpret_cast<const uint4*>(bl + off)) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int k = 0; k < 3; ++k) gv[u][k] = (ok && k < nc) ? __ldg(job.g + m * job.gs + k) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float x[8];
        unpack8(vh[u], vl[u], x);
        if (nc == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] += x[i];
        } else {
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            if (k < nc) {
#pragma unroll
              for (int i = 0; i < 8; ++i) acc[k * 8 + i] = fmaf(gv[u][k], x[i], acc[k * 8 + i]);
              if (c16 == 0) accb[k] += gv[u][k];
            }
          }
        }
      }
    }
  }
  const int nk = nc == 0 ? 1 : nc;
  for (int k = 0; k < nk; ++k)
#pragma unroll
    for (int i = 0; i < 8; ++i) red[rg][c16][k * 8 + i] = acc[k * 8 + i];
  if (c16 == 0) red[rg][0][24] = 0.f;
  __syncthreads();
  // 256 threads: thread -> (feature chunk c16', element i) for k = 0.. ; sum over the 8 row groups
  for (int idx = tid; idx < 32 * 8 * nk; idx += 256) {
    const int k = idx / 256, rem = idx % 256, cc = rem >> 3, i = rem & 7;
    if ((cc >> 3) >= job.nblk) continue;
    float v = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) v += red[r][cc][k * 8 + i];
    atomicAdd(job.out + (size_t)k * job.ldo + cc * 8 + i, v);
  }
  if (nc > 0 && job.out_bias) {
    __syncthreads();
    if (c16 == 0) { red[rg][0][0] = accb[0]; red[rg][0][1] = accb[1]; red[rg][0][2] = accb[2]; }
    __syncthreads();
    if (tid < nc) {
      float v = 0.f;
      for (int r = 0; r < 8; ++r) v += red[r][0][tid];
      atomicAdd(job.out_bias + tid, v);
    }
  }
}

// per-ray sum of g_hid over the samples: rayS[r][n] = sum_k GHID[(r,k)][n].  Block = one ray, 128 threads =
// 8 sample groups x 16 sixteen-byte chunks (8 features each), reduced through shared memory.
__global__ void __launch_bounds__(128) ray_sum_ghid_kernel(Images img, int R, int S, float* __restrict__ rayS) {
  __shared__ float red[8][128];
  const int r = blockIdx.x, c = threadIdx.x & 15, g = threadIdx.x >> 4;   // chunk c: features 8c..8c+7
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int k = g; k < S; k += 8) {
    const long long m = (long long)r * S + k;
    const int tile = (int)(m >> 7), row = (int)(m & 127);
    const uint32_t off = sw128_offset(row, (c & 7) * 8);
    float x[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(img.at(T_GHID, tile, c >> 3, 0) + off)),
            __ldg(reinterpret_cast<const uint4*>(img.at(T_GHID, tile, c >> 3, 1) + off)), x);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] += x[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[g][c * 8 + i] = acc[i];
  __syncthreads();
  float v = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) v += red[q][threadIdx.x];
  rayS[(size_t)r * kHW + threadIdx.x] = v;
}

// view-direction part of the colour head: dW8[n][256+k] += sum_r rayS[r][n] denc[r][k]
__global__ void ray_head_wgrad_kernel(int R, int rays_per_block, const float* __restrict__ rayS,
                                      const float* __restrict__ denc, float* __restrict__ dW8) {
  const int n = threadIdx.x;   // 128
  const int r0 = blockIdx.x * rays_per_block, r1 = min(R, r0 + rays_per_block);
  float acc[kEv];
#pragma unroll
  for (int k = 0; k < kEv; ++k) acc[k] = 0.f;
  for (int r = r0; r < r1; ++r) {
    const float s = rayS[(size_t)r * kHW + n];
#pragma unroll
    for (int k = 0; k < kEv; ++k) acc[k] = fmaf(s, denc[(size_t)r * 32 + k], acc[k]);
  }
#pragma unroll
  for (int k = 0; k < kEv; ++k) atomicAdd(dW8 + (size_t)n * (kW + kEv) + kW + k, acc[k]);
}

// ------------------------------------------------------------------------------------------------
// ray gradients (camera-pose optimisation): dL/d enc = G4 . W4[:, 256:319] + G0 . W0 on tensor cores, then the
// positional-encoding backward and the reduction over each ray's samples in the epilogue.
//   d/dx [w sin(f x)] = f * (w cos(f x)) = f * enc_cos ;  d/dx [w cos(f x)] = -f * enc_sin
// ------------------------------------------------------------------------------------------------
constexpr int kEgStages = 3;
constexpr int kEgWBytes = 16 * 8192;                         // 2 layers x 4 K blocks x (hi, lo) x [64 x 64]
constexpr int kEgStageBytes = 2 * kChunkBytes;               // one K block of G: hi + lo
constexpr int kEgSmem = kEgWBytes + kEgStages * kEgStageBytes + 256;

// chunk (li in {0: layer 4 skip columns, 1: layer 0}, kb, part): [64 (n = internal encoder column) x 64 (k = out feature)]
__global__ void pack_weights_enc_kernel(const float* __restrict__ w4, const float* __restrict__ w0, uint8_t* __restrict__ packed) {
  const int chunk = blockIdx.x;              // (li * 4 + kb) * 2 + part
  const int part = chunk & 1, kb = (chunk >> 1) & 3, li = chunk >> 3;
  const float* W = li == 0 ? w4 : w0;
  const int ldw = li == 0 ? kW + 63 : 63, colbase = li == 0 ? kW : 0;
  uint8_t* dst = packed + (size_t)chunk * 8192;
  for (int e = threadIdx.x; e < 64 * 64; e += blockDim.x) {
    const int n = e >> 6, k = e & 63;
    const int rc = enc_ref_col(n);
    const float v = rc < 0 ? 0.f : W[(size_t)(kb * 64 + k) * ldw + colbase + rc];
    *reinterpret_cast<uint16_t*>(dst + sw128_offset(n, k)) = split1<false>(v, part);
  }
}

struct EncGradParams {
  const uint8_t* packed;      // 16 chunks of 8 KB
  Images img;
  const float* t;             // [M]
  float* d_origins;           // [R,3] (+=), may be NULL
  float* d_dirs;              // [R,3] (+=), may be NULL
  long long M;
  int S, num_tiles;
};

__global__ void __launch_bounds__(192, 1) tc_mlp_encgrad_kernel(const EncGradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_w = smem;
  uint8_t* s_a = smem + kEgWBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_a + kEgStages * kEgStageBytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + kEgStages;
  uint64_t* w_ready = bars + 2 * kEgStages;
  uint64_t* d_full = w_ready + 1;
  uint64_t* d_empty = w_ready + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_ready + 3);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < kEgStages; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    mbar_init(w_ready, 1);
    mbar_init(d_full, 1);
    mbar_init(d_empty, 4);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 64);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(w_ready, kEgWBytes);
      for (int c = 0; c < 16; ++c) bulk_g2s(s_w + c * 8192, p.packed + (size_t)c * 8192, 8192, w_ready);
      uint32_t stage = 0, phase = 0;
      for (int it = 0; it < my_tiles; ++it) {
        const int tile = blockIdx.x + it * gridDim.x;
        for (int li = 0; li < 2; ++li) {
          const int tg = li == 0 ? t_g(4) : t_g(0);
          for (int kb = 0; kb < 4; ++kb) {
            mbar_wait(&a_empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&a_full[stage], kEgStageBytes);
            bulk_g2s(s_a + stage * kEgStageBytes, p.img.at(tg, tile, kb, 0), kChunkBytes, &a_full[stage]);
            bulk_g2s(s_a + stage * kEgStageBytes + kChunkBytes, p.img.at(tg, tile, kb, 1), kChunkBytes, &a_full[stage]);
            if (++stage == kEgStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(128, 64, 1);
      mbar_wait(w_ready, 0);
      tc_fence_after();
      uint32_t stage = 0, phase = 0;
      for (int it = 0; it < my_tiles; ++it) {
        mbar_wait(d_empty, (it & 1) ^ 1);
        tc_fence_after();
        for (int li = 0; li < 2; ++li) {
          for (int kb = 0; kb < 4; ++kb) {
            mbar_wait(&a_full[stage], phase);
            tc_fence_after();
            const uint32_t a_hi = smem_u32(s_a + stage * kEgStageBytes), a_lo = a_hi + kChunkBytes;
            const uint32_t w_hi = smem_u32(s_w + ((li * 4 + kb) * 2) * 8192), w_lo = w_hi + 8192;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              umma_ss(tmem_base, make_smem_desc(a_hi + ks * 32), make_smem_desc(w_hi + ks * 32), idesc, (li | kb | ks) != 0);
              umma_ss(tmem_base, make_smem_desc(a_lo + ks * 32), make_smem_desc(w_hi + ks * 32), idesc, 1u);
              umma_ss(tmem_base, make_smem_desc(a_hi + ks * 32), make_smem_desc(w_lo + ks * 32), idesc, 1u);
            }
            umma_commit(&a_empty[stage]);
            if (++stage == kEgStages) { stage = 0; phase ^= 1; }
          }
        }
        umma_commit(d_full);
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    for (int it = 0; it < my_tiles; ++it) {
      const int tile = blockIdx.x + it * gridDim.x;
      const long long m = (long long)tile * kTileM + row;
      const bool valid = m < p.M;
      mbar_wait(d_full, it & 1);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16), v0);
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(d_empty);
      // encoder values of this row (hi + lo image), internal column order
      float gx[3] = {0.f, 0.f, 0.f};
      {
        const uint8_t* eh = p.img.at(T_ENC, tile, 0, 0);
        const uint8_t* el = p.img.at(T_ENC, tile, 0, 1);
        float g[64];
#pragma unroll
        for (int i = 0; i < 32; ++i) { g[i] = __uint_as_float(v0[i]); g[32 + i] = __uint_as_float(v1[i]); }
        gx[0] = g[0]; gx[1] = g[1]; gx[2] = g[2];
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          float e[8];
          const uint32_t off = sw128_offset(row, c8 * 8);
          unpack8(*reinterpret_cast<const uint4*>(eh + off), *reinterpret_cast<const uint4*>(el + off), e);
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const int ic = c8 * 8 + i;               // (sin, cos) pair at internal columns ic, ic+1 (ic >= 4)
            if (ic < 4) continue;
            const int pr = (ic - 4) >> 1, c = pr / kL, j = pr - c * kL;
            const float f = band_freq(j);
            const float contrib = f * (g[ic] * e[i + 1] - g[ic + 1] * e[i]);
            if (c == 0) gx[0] += contrib; else if (c == 1) gx[1] += contrib; else gx[2] += contrib;
          }
        }
      }
      const float tv = valid ? p.t[m] : 0.f;
      float so[3], sd[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) { so[c] = valid ? gx[c] : 0.f; sd[c] = so[c] * tv; }
      // rows of one warp usually belong to one ray (S multiple of 32): reduce before the atomics
      const long long ray = valid ? m / p.S : -1;
      const long long ray0 = __shfl_sync(0xffffffffu, ray, 0);
      const bool uniform = __all_sync(0xffffffffu, ray == ray0);
      if (uniform) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
          for (int s = 16; s > 0; s >>= 1) {
            so[c] += __shfl_xor_sync(0xffffffffu, so[c], s);
            sd[c] += __shfl_xor_sync(0xffffffffu, sd[c], s);
          }
        }
        if (lane == 0 && ray0 >= 0) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if (p.d_origins) atomicAdd(p.d_origins + ray0 * 3 + c, so[c]);
            if (p.d_dirs) atomicAdd(p.d_dirs + ray0 * 3 + c, sd[c]);
          }
        }
      } else if (valid) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if (p.d_origins) atomicAdd(p.d_origins + ray * 3 + c, so[c]);
          if (p.d_dirs) atomicAdd(p.d_dirs + ray * 3 + c, sd[c]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 64);
}

// view-direction part: Gdenc[r][k] = sum_n rayS[r][n] * W8[n][256 + k]
__global__ void ray_head_dgrad_kernel(int R, const float* __restrict__ rayS, const float* __restrict__ w8,
                                      float* __restrict__ gdenc) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= R * 32) return;
  const int r = idx >> 5, k = idx & 31;
  float acc = 0.f;
  if (k < kEv)
    for (int n = 0; n < kHW; ++n) acc = fmaf(rayS[(size_t)r * kHW + n], w8[(size_t)n * (kW + kEv) + kW + k], acc);
  gdenc[idx] = acc;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool tc_supports(const SparfMLP* mlp) {
  return mlp && mlp->n_trunk == 8 && mlp->width == kW && mlp->head_width == kHW && mlp->skip_layer == 4 &&
         mlp->L_xyz == kL && mlp->L_view == kLv;
}

static int tape_tiles(int R, int S);
static size_t tape_off_denc(int R, int S);
static size_t tape_off_packed_b(int R, int S);
static size_t tape_off_packed_e(int R, int S);

// rays per backward chunk: <= 1024 row tiles of gradient images (~1.1 GB), a whole number of 128-row tiles (a taped
// forward numbers its tiles over the whole batch, so every chunk has to start on a tile boundary)
static int gcd_int(int a, int b) { return b == 0 ? a : gcd_int(b, a % b); }
static int bwd_chunk_rays(int S) {
  const int unit = kTileM / gcd_int(S, kTileM);          // smallest ray count whose rows fill whole tiles
  const int n = (1024 * kTileM) / S;
  return std::max(unit, n - n % unit);
}

static size_t images_bytes(int ntiles, int t_begin, int t_end) {
  size_t total = 0;
  for (int t = t_begin; t < t_end; ++t) total += (size_t)tensor_nblk(t) * 2 * kChunkBytes * ntiles;
  return total;
}
static size_t fwd_images_bytes(int ntiles) { return images_bytes(ntiles, 0, T_GHID) + (size_t)ntiles * kMaskTileBytes; }
static size_t bwd_images_bytes(int ntiles) { return images_bytes(ntiles, T_GHID, T_COUNT); }
// Forward tensors: laid out for `ntiles_fwd` tiles, the returned pointers address tile `tile0` of each (a backward chunk
// of a larger taped batch); gradient tensors: `ntiles_bwd` tiles of the chunk's own workspace.
static void images_assign(Images& img, int ntiles_fwd, uint8_t* fwd_base, uint8_t* bwd_base, int tile0 = 0, int ntiles_bwd = -1) {
  if (ntiles_bwd < 0) ntiles_bwd = ntiles_fwd;
  size_t o = 0;
  for (int t = 0; t < T_GHID; ++t) {
    const size_t per_tile = (size_t)tensor_nblk(t) * 2 * kChunkBytes;
    img.ptr[t] = fwd_base ? fwd_base + o + per_tile * tile0 : nullptr;
    o += per_tile * ntiles_fwd;
  }
  img.mask = fwd_base ? fwd_base + o + kMaskTileBytes * tile0 : nullptr;
  o = 0;
  for (int t = T_GHID; t < T_COUNT; ++t) { img.ptr[t] = bwd_base ? bwd_base + o : nullptr; o += (size_t)tensor_nblk(t) * 2 * kChunkBytes * ntiles_bwd; }
}

struct BwdCarve {
  uint8_t *packed_f, *packed_b, *images_f, *images_b;
  float *raybias, *denc, *sigma, *rgb, *g_raw, *g_pre, *rayS, *gdenc;
  uint8_t* packed_e;
  size_t total;
};

static BwdCarve bwd_carve(void* ws, int nr, int S, bool with_fwd_images) {
  const size_t Mc = (size_t)nr * S;
  const int ntiles = (int)((Mc + kTileM - 1) / kTileM);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 1024); return r; };
  BwdCarve c;
  uint8_t* b = reinterpret_cast<uint8_t*>(ws);
  size_t o_pf = take((size_t)kChunksPerTile * kChunkBytes), o_pb = take((size_t)kBwdChunksPerTile * kChunkBytes);
  size_t o_rb = take((size_t)nr * kHW * 4), o_de = take((size_t)nr * 32 * 4), o_si = take(Mc * 4), o_rg = take(Mc * 12);
  size_t o_gr = take(Mc * 4), o_gp = take(Mc * 16), o_rs = take((size_t)nr * kHW * 4);
  size_t o_gd = take((size_t)nr * 32 * 4), o_pe = take(kEgWBytes);
  size_t o_ib = take(bwd_images_bytes(ntiles));
  size_t o_if = take(with_fwd_images ? fwd_images_bytes(ntiles) : 0);
  c.packed_f = b + o_pf; c.packed_b = b + o_pb; c.raybias = (float*)(b + o_rb); c.denc = (float*)(b + o_de);
  c.sigma = (float*)(b + o_si); c.rgb = (float*)(b + o_rg); c.g_raw = (float*)(b + o_gr); c.g_pre = (float*)(b + o_gp);
  c.rayS = (float*)(b + o_rs); c.gdenc = (float*)(b + o_gd); c.packed_e = b + o_pe; c.images_b = b + o_ib; c.images_f = with_fwd_images ? b + o_if : nullptr;
  c.total = o + 1024;
  return c;
}

// forward workspace (inference and taped forward): packed forward weight stream | raybias [R,128]
struct FwdCarve {
  uint8_t* packed;
  float* raybias;
  size_t total;
};

static FwdCarve fwd_carve(void* ws, int R) {
  const size_t o_rb = align_up((size_t)kChunksPerTile * kChunkBytes, 256);
  FwdCarve c;
  c.packed = reinterpret_cast<uint8_t*>(ws);
  c.raybias = reinterpret_cast<float*>(c.packed + o_rb);
  c.total = o_rb + align_up((size_t)R * kHW * sizeof(float), 256) + 256;
  return c;
}

size_t tc_workspace_bytes(const SparfMLP* mlp, int R, int S, int backward, int engine) {
  if (backward) {   // 1: recompute path (forward images of a chunk live in the workspace); 2: a tape holds them
    int nr = std::min(R, bwd_chunk_rays(S));
    return bwd_carve(nullptr, nr, S, backward != 2).total;
  }
  return fwd_carve(nullptr, R).total;
}

static void fill_pack_params(const SparfMLP* mlp, PackParams& pp, uint8_t* dst) {
  for (int l = 0; l < 8; ++l) pp.w[l] = mlp->trunk_w[l];
  pp.w[8] = mlp->head_w[0];
  pp.packed = dst;
  pp.order = 0;
}

// which forward kernel serves a call: the A operand in tensor memory for fp16 3-pass calls (every default call), operands
// in shared memory otherwise (single-pass engine, bf16 recompute forward).  The weight packing order follows it.
static bool fwd_tmem(bool f16, int passes) { return f16 && passes == 3; }

#ifdef SPARF_TC_TRACE
static void trace_dump(const char* what) {
  static long long h[148 * 6 * 8];
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(h, g_tc_trace, sizeof(h));
  const char* roles[5] = {"producer0 (w0 = ring slot free)", "mma issuer (w0 = acc free, w1 = A ready, w2 = weights landed)",
                          "epilogue warp 0 (w0 = acc full; fwd: w1 = staging slot free, w2 = tmem ld, w3 = encoding; dgrad: w1 = mask loads, w2 = tmem ld, w3 = staging slot free)",
                          "epilogue warp 15", "image store warp (w0 = block staged, w1 = bulk store issue + source read)"};
  fprintf(stderr, "[tc trace] %s, mean over CTAs 0..147 (clocks)\n", what);
  for (int r = 0; r < 5; ++r) {
    double a[5] = {0, 0, 0, 0, 0};
    for (int b = 0; b < 148; ++b)
      for (int k = 0; k < 5; ++k) a[k] += (double)h[((size_t)b * 6 + r) * 8 + k] / 148.0;
    fprintf(stderr, "  %-70s total %9.0f  w0 %9.0f  w1 %9.0f  w2 %9.0f  w3 %9.0f\n", roles[r], a[4], a[0], a[1], a[2], a[3]);
  }
  if (getenv("SPARF_TC_TRACE_EVENTS")) {
    static long long ev[512 * 8];
    cudaMemcpyFromSymbol(ev, g_tc_events, sizeof(ev));
    const long long t0 = ev[1];
    fprintf(stderr, "  chunk: slot-free  copy-issued | issuer: at-wait  weights-seen  mmas-issued  committed   (clocks since first copy)\n");
    for (int g = 128; g < 200; ++g)
      fprintf(stderr, "  %4d: %9lld %9lld | %9lld %9lld %9lld %9lld\n", g, ev[g * 8] - t0, ev[g * 8 + 1] - t0, ev[g * 8 + 2] - t0,
              ev[g * 8 + 3] - t0, ev[g * 8 + 4] - t0, ev[g * 8 + 5] - t0);
  }
}
#define TRACE_DUMP(what) trace_dump(what)
#else
#define TRACE_DUMP(what) ((void)0)
#endif

static int launch_forward(const SparfMLP* mlp, bool f16, int passes, int nr, int S, const float* origins, const float* dirs,
                          const float* t, const float* noise, float* sigma, float* rgb, const uint8_t* packed,
                          const float* raybias, const Images* img, cudaStream_t st, int save_mode = 1) {
  FwdParams p;
  p.packed = packed;
  p.raybias = raybias;
  p.origins = origins; p.dirs = dirs; p.t = t; p.noise = noise;
  p.sigma = sigma; p.rgb = rgb;
  for (int l = 0; l < 8; ++l) p.bias[l] = mlp->trunk_b[l];
  p.w7 = mlp->trunk_w[7];
  p.w9 = mlp->head_w[1];
  p.b9 = mlp->head_b[1];
  p.c2f = C2F{mlp->use_c2f, mlp->c2f_start, mlp->c2f_range, mlp->progress};
  p.M = (long long)nr * S;
  p.S = S;
  p.num_tiles = (int)((p.M + kTileM - 1) / kTileM);
  p.passes = passes;
  p.save = img != nullptr ? save_mode : 0;
  if (img) p.img = *img; else { for (int i = 0; i < T_COUNT; ++i) p.img.ptr[i] = nullptr; }
  static bool attr_set_dev[64] = {};
  int dev_ord = 0;
  cudaGetDevice(&dev_ord);
  bool& attr_set = attr_set_dev[dev_ord & 63];   // function attributes are per device
  if (!attr_set) {
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_fwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_fwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_fwd_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_fwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem + 1024));
    SPARF_CHECK_CUDA(cudaFuncSetAttribute(tc_mlp_encgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kEgSmem + 1024));
    attr_set = true;
  }
  const bool tmem = fwd_tmem(f16, passes);
  if (!tmem && p.save == 2) p.save = 1;     // the shared-memory-operand kernels always write both halves
  if (tmem && p.save == 2) {
    tc_mlp_fwd_kernel<true, true, true><<<std::min(p.num_tiles, num_sms()), kThreads, kSmemBytes + 1024, st>>>(p);
    TRACE_DUMP("forward (hi-only tape, A in TMEM)");
  } else if (tmem) {
    tc_mlp_fwd_kernel<true, true><<<std::min(p.num_tiles, num_sms()), kThreads, kSmemBytes + 1024, st>>>(p);
    TRACE_DUMP(p.save ? "forward (tape, A in TMEM)" : "forward f16 (A in TMEM)");
  } else {
    int grid = std::min(p.num_tiles, num_sms());
    if (f16) tc_mlp_fwd_kernel<true, false><<<grid, kThreads, kSmemBytes + 1024, st>>>(p);
    else tc_mlp_fwd_kernel<false, false><<<grid, kThreads, kSmemBytes + 1024, st>>>(p);
    TRACE_DUMP(p.save ? "forward (tape)" : (f16 ? "forward f16" : "forward bf16"));
  }
  SPARF_CHECK_LAUNCH("tc_mlp_fwd_kernel");
  return SPARF_OK;
}

int tc_mlp_forward(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                   const float* t, const float* noise, float* sigma, float* rgb, void* workspace,
                   size_t workspace_bytes, cudaStream_t st) {
  int rc = simt_validate(mlp);
  if (rc) return rc;
  if (!tc_supports(mlp)) {
    set_error("tcgen05 engine: unsupported MLP shape (needs 8x256 trunk, skip 4, L_xyz=10, L_view=4, head 128)");
    return SPARF_ERR_UNSUPPORTED;
  }
  if (workspace_bytes < tc_workspace_bytes(mlp, R, S, 0, engine)) {
    set_error("tc_mlp_forward: workspace %zu < %zu bytes", workspace_bytes, tc_workspace_bytes(mlp, R, S, 0, engine));
    return SPARF_ERR_WORKSPACE;
  }
  const FwdCarve ws = fwd_carve(workspace, R);
  const int passes = engine == SPARF_ENGINE_TC_1X ? 1 : 3;
  PackParams pp;
  fill_pack_params(mlp, pp, ws.packed);
  pp.order = fwd_tmem(true, passes) ? 1 : 0;
  pack_weights_kernel<true><<<kChunksPerTile, 1024, 0, st>>>(pp);   // one element group per thread
  SPARF_CHECK_LAUNCH("pack_weights_kernel");
  C2F c2f{mlp->use_c2f, mlp->c2f_start, mlp->c2f_range, mlp->progress};
  raybias_kernel<<<ceil_div(R, 4), 512, 0, st>>>(R, dirs, mlp->head_w[0], mlp->head_b[0], c2f, ws.raybias, nullptr);
  SPARF_CHECK_LAUNCH("raybias_kernel");
  return launch_forward(mlp, true, passes, R, S, origins, dirs, t, noise, sigma, rgb, ws.packed, ws.raybias, nullptr, st);
}

// Fork / join onto a library-owned side stream (one per device, created on first use): the CUDA-core leftovers of the
// backward (bias / narrow-layer reductions, view-direction columns, ray gradients) only depend on the dgrad chain, so
// they run BESIDE the HBM-bound weight-gradient kernel instead of after it (its CTAs leave ~30 KB of shared memory and
// most thread slots of every SM free).  Event record / wait pairs make the pattern capturable into a CUDA graph.
struct SideStream {
  bool ready = false;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr, stream3 = nullptr;   // backward leftovers: three independent chains beside the wgrad kernel
  cudaEvent_t join2 = nullptr, join3 = nullptr, rayhead = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaEvent_t raybias = nullptr, packed = nullptr;   // taped forward: raybias ready / backward weight streams packed
};
// nullptr (with the error text set) if the streams or events cannot be created
static SideStream* side_stream() {
  static SideStream table[64];
  int dev = 0;
  cudaGetDevice(&dev);
  SideStream& s = table[dev & 63];
  if (!s.ready) {
    cudaError_t e = cudaSuccess;
    for (cudaStream_t* p : {&s.stream, &s.stream2, &s.stream3})
      if (e == cudaSuccess && !*p) e = cudaStreamCreateWithFlags(p, cudaStreamNonBlocking);
    for (cudaEvent_t* p : {&s.join2, &s.join3, &s.rayhead, &s.fork, &s.join, &s.raybias, &s.packed})
      if (e == cudaSuccess && !*p) e = cudaEventCreateWithFlags(p, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      set_error("tcgen05 engine: cannot create its side streams: %s", cudaGetErrorString(e));
      return nullptr;
    }
    s.ready = true;
  }
  return &s;
}

// Training forward: same fp16-split arithmetic and outputs as tc_mlp_forward, plus the tape for the backward.
int tc_mlp_forward_tape(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                        const float* t, const float* noise, float* sigma, float* rgb, void* tape, size_t tape_bytes,
                        void* workspace, size_t workspace_bytes, cudaStream_t st) {
  int rc = simt_validate(mlp);
  if (rc) return rc;
  const size_t need = tc_tape_bytes(mlp, R, S);
  if (need == 0 || tape == nullptr || tape_bytes < need) {
    set_error("tc_mlp_forward_tape: tape unsupported for this call or too small (%zu < %zu bytes)", tape_bytes, need);
    return SPARF_ERR_WORKSPACE;
  }
  if (workspace_bytes < tc_workspace_bytes(mlp, R, S, 0, engine)) {
    set_error("tc_mlp_forward_tape: workspace %zu < %zu bytes", workspace_bytes, tc_workspace_bytes(mlp, R, S, 0, engine));
    return SPARF_ERR_WORKSPACE;
  }
  const FwdCarve ws = fwd_carve(workspace, R);
  const int ntiles = tape_tiles(R, S);
  uint8_t* tp = reinterpret_cast<uint8_t*>(tape);
  float* denc = reinterpret_cast<float*>(tp + tape_off_denc(R, S));
  C2F c2f{mlp->use_c2f, mlp->c2f_start, mlp->c2f_range, mlp->progress};
  // side stream: the per-ray colour-head bias (needed by the forward kernel) and the two weight streams of the
  // BACKWARD (needed only by sparf_mlp_backward_tape) run beside the forward packing / kernel
  SideStream* side = side_stream();
  if (!side) return SPARF_ERR_CUDA;
  SPARF_CHECK_CUDA(cudaEventRecord(side->fork, st));
  SPARF_CHECK_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
  raybias_kernel<<<ceil_div(R, 4), 512, 0, side->stream>>>(R, dirs, mlp->head_w[0], mlp->head_b[0], c2f, ws.raybias, denc);
  SPARF_CHECK_LAUNCH("raybias_kernel");
  SPARF_CHECK_CUDA(cudaEventRecord(side->raybias, side->stream));
  PackParams pp;
  fill_pack_params(mlp, pp, ws.packed);
  pp.order = fwd_tmem(true, 3) ? 1 : 0;
  pack_weights_kernel<true><<<kChunksPerTile, 1024, 0, st>>>(pp);   // on the forward's critical path: one element group
                                                                      // per thread (13 -> ~6 us)
  SPARF_CHECK_LAUNCH("pack_weights_kernel");
  PackParams pb;
  fill_pack_params(mlp, pb, tp + tape_off_packed_b(R, S));
  pack_weights_bwd_kernel<<<kBwdChunksPerTile, 256, 0, side->stream>>>(pb);
  SPARF_CHECK_LAUNCH("pack_weights_bwd_kernel");
  pack_weights_enc_kernel<<<16, 256, 0, side->stream>>>(mlp->trunk_w[4], mlp->trunk_w[0], tp + tape_off_packed_e(R, S));
  SPARF_CHECK_LAUNCH("pack_weights_enc_kernel");
  SPARF_CHECK_CUDA(cudaEventRecord(side->packed, side->stream));
  SPARF_CHECK_CUDA(cudaStreamWaitEvent(st, side->raybias, 0));
  Images img;
  images_assign(img, ntiles, tp, nullptr);
  // TC_3X_W1: the weight gradients will take the hi halves only, so only those are written (the tape keeps its layout)
  rc = launch_forward(mlp, true, 3, R, S, origins, dirs, t, noise, sigma, rgb, ws.packed, ws.raybias, &img, st,
                      engine == SPARF_ENGINE_TC_3X_W1 ? 2 : 1);
  // join: whatever follows on the caller's stream (the backward, or a reuse of the tape's memory) is ordered after the
  // side-stream packing, which has long finished by the time the forward kernel ends
  if (rc == SPARF_OK) SPARF_CHECK_CUDA(cudaStreamWaitEvent(st, side->packed, 0));
  return rc;
}

// tape = what the training forward keeps for the backward: the forward operand images of every row tile
// followed by the per-ray view-direction encoding [R,32]
static int tape_tiles(int R, int S) { return (int)(((long long)R * S + kTileM - 1) / kTileM); }
constexpr size_t kMaxTapeBytes = (size_t)64 << 30;   // beyond this the backward recomputes the forward chunk by chunk
// tape = forward operand images | per-ray view-direction encoding [R,32] | backward weight stream (120 x 16 KB) |
//        ray-gradient weight stream (128 KB): the two packed streams are produced by the FORWARD call on the side
//        stream, beside the forward kernel, so the backward starts with its dgrad chain
static size_t tape_off_denc(int R, int S) { return align_up(fwd_images_bytes(tape_tiles(R, S)), 1024); }
static size_t tape_off_packed_b(int R, int S) { return tape_off_denc(R, S) + align_up((size_t)R * 32 * 4, 1024); }
static size_t tape_off_packed_e(int R, int S) { return tape_off_packed_b(R, S) + (size_t)kBwdChunksPerTile * kChunkBytes; }
size_t tc_tape_bytes(const SparfMLP* mlp, int R, int S) {
  if (!tc_supports(mlp)) return 0;
  const size_t need = tape_off_packed_e(R, S) + kEgWBytes;
  return need <= kMaxTapeBytes ? need : 0;
}

static int tc_mlp_backward_impl(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                                const float* t, const float* noise, const float* d_sigma, const float* d_rgb,
                                const SparfMLPGrad* grad, float* d_origins, float* d_dirs, void* workspace,
                                size_t workspace_bytes, uint8_t* tape, const float* sigma_fwd, const float* rgb_fwd,
                                cudaStream_t st);

int tc_mlp_backward(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                    const float* t, const float* noise, const float* d_sigma, const float* d_rgb,
                    const SparfMLPGrad* grad, float* d_origins, float* d_dirs, void* workspace,
                    size_t workspace_bytes, cudaStream_t st) {
  return tc_mlp_backward_impl(mlp, engine, R, S, origins, dirs, t, noise, d_sigma, d_rgb, grad, d_origins, d_dirs, workspace,
                              workspace_bytes, nullptr, nullptr, nullptr, st);
}

int tc_mlp_backward_tape(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                         const float* t, const float* sigma, const float* rgb, const float* d_sigma, const float* d_rgb,
                         const SparfMLPGrad* grad, float* d_origins, float* d_dirs, void* tape, size_t tape_bytes,
                         void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (tape == nullptr || tape_bytes < tc_tape_bytes(mlp, R, S) || tc_tape_bytes(mlp, R, S) == 0) {
    set_error("tc_mlp_backward_tape: tape missing or too small (%zu < %zu bytes)", tape_bytes, tc_tape_bytes(mlp, R, S));
    return SPARF_ERR_WORKSPACE;
  }
  return tc_mlp_backward_impl(mlp, engine, R, S, origins, dirs, t, nullptr, d_sigma, d_rgb, grad, d_origins, d_dirs, workspace,
                              workspace_bytes, reinterpret_cast<uint8_t*>(tape), sigma, rgb, st);
}

static int tc_mlp_backward_impl(const SparfMLP* mlp, int engine, int R, int S, const float* origins, const float* dirs,
                                const float* t, const float* noise, const float* d_sigma, const float* d_rgb,
                                const SparfMLPGrad* grad, float* d_origins, float* d_dirs, void* workspace,
                                size_t workspace_bytes, uint8_t* tape, const float* sigma_fwd, const float* rgb_fwd,
                                cudaStream_t st) {
  int rc = simt_validate(mlp);
  if (rc) return rc;
  if (!tc_supports(mlp)) {
    set_error("tcgen05 engine: unsupported MLP shape");
    return SPARF_ERR_UNSUPPORTED;
  }
  if (workspace_bytes < tc_workspace_bytes(mlp, R, S, tape ? 2 : 1, engine)) {
    set_error("tc_mlp_backward: workspace %zu < %zu bytes", workspace_bytes, tc_workspace_bytes(mlp, R, S, tape ? 2 : 1, engine));
    return SPARF_ERR_WORKSPACE;
  }
  SideStream* side = side_stream();
  if (!side) return SPARF_ERR_CUDA;
  const int nrc = std::min(R, bwd_chunk_rays(S));
  const C2F c2f{mlp->use_c2f, mlp->c2f_start, mlp->c2f_range, mlp->progress};
  for (int r0 = 0; r0 < R; r0 += nrc) {
    const int nr = std::min(nrc, R - r0);
    const long long Mc = (long long)nr * S;
    const size_t m0 = (size_t)r0 * S;
    const int ntiles = (int)((Mc + kTileM - 1) / kTileM);
    BwdCarve c = bwd_carve(workspace, nr, S, tape == nullptr);
    Images img;
    if (tape) {   // forward images + denc + forward outputs of the whole batch come from the tape; this chunk = tiles
                  // [m0 / 128, ...) of it (bwd_chunk_rays keeps every chunk on a tile boundary)
      const int ntiles_all = tape_tiles(R, S);
      images_assign(img, ntiles_all, tape, c.images_b, (int)(m0 / kTileM), ntiles);
      c.denc = reinterpret_cast<float*>(tape + tape_off_denc(R, S)) + (size_t)r0 * 32;
      c.packed_b = tape + tape_off_packed_b(R, S);      // packed by the forward call (side stream)
      c.packed_e = tape + tape_off_packed_e(R, S);
      c.sigma = const_cast<float*>(sigma_fwd) + m0;
      c.rgb = const_cast<float*>(rgb_fwd) + m0 * 3;
    } else {
      images_assign(img, ntiles, c.images_f, c.images_b);
    }

    PackParams pp;
    if (!tape) {
      fill_pack_params(mlp, pp, c.packed_f);
      pack_weights_kernel<false><<<kChunksPerTile, 256, 0, st>>>(pp);
      SPARF_CHECK_LAUNCH("pack_weights_kernel<bf16>");
    }
    if (!tape) {
      fill_pack_params(mlp, pp, c.packed_b);
      pack_weights_bwd_kernel<<<kBwdChunksPerTile, 256, 0, st>>>(pp);
      SPARF_CHECK_LAUNCH("pack_weights_bwd_kernel");
    }   // (with a tape the forward call packed both backward weight streams on the side stream and joined)
    if (!tape) {
      raybias_kernel<<<ceil_div(nr, 4), 512, 0, st>>>(nr, dirs + (size_t)r0 * 3, mlp->head_w[0], mlp->head_b[0], c2f, c.raybias, c.denc);
      SPARF_CHECK_LAUNCH("raybias_kernel");
      // 1. forward re-run (bf16 halves) dumping the operand images
      rc = launch_forward(mlp, false, 3, nr, S, origins + (size_t)r0 * 3, dirs + (size_t)r0 * 3, t + m0,
                          noise ? noise + m0 : nullptr, c.sigma, c.rgb, c.packed_f, c.raybias, &img, st);
      if (rc) return rc;
    }

    // 2. input-gradient chain
    const int wg_passes = engine == SPARF_ENGINE_TC_3X_W1 ? 1 : 3;
    BwdParams bp;
    bp.hi_only = wg_passes == 1;
    bp.packed = c.packed_b;
    bp.d_sigma = d_sigma + m0; bp.d_rgb = d_rgb + m0 * 3;
    bp.sigma = c.sigma; bp.rgb = c.rgb;
    bp.g_raw = c.g_raw; bp.g_pre = c.g_pre;
    bp.w7 = mlp->trunk_w[7]; bp.w9 = mlp->head_w[1];
    bp.M = Mc; bp.num_tiles = ntiles; bp.img = img;
    // A operand in tensor memory (shared-memory operands measured 360 vs 294 us, profiles/r02_notes.md)
    tc_mlp_dgrad_kernel<<<std::min(ntiles, num_sms()), kThreads, kSmemBytes + 1024, st>>>(bp);
    TRACE_DUMP("dgrad");
    SPARF_CHECK_LAUNCH("tc_mlp_dgrad_kernel");

    // fork: the CUDA-core leftovers (steps 4, 5) run on the side streams beside the weight-gradient kernel
    SPARF_CHECK_CUDA(cudaEventRecord(side->fork, st));
    SPARF_CHECK_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    cudaStream_t sd = side->stream, sd2 = side->stream, sd3 = side->stream;
    // Up to three independent chains, so that together they are shorter than the weight-gradient kernel they run beside
    // (each is slowed down several-fold while it shares the GPU with it).  With ray gradients the leftovers
    // (reductions + ray-gradient GEMM + view-direction chain) are longer than the weight-gradient kernel when serialised:
    // three chains (c3: 4.46 -> 4.39 ms); without them one chain is enough and measured marginally faster (c2: 1.335 vs
    // 1.345 ms).  (The single-pass weight-gradient kernel is short enough that the serial chain outlasts it even without
    // them.)
    if (d_origins != nullptr || d_dirs != nullptr || wg_passes == 1) {
      SPARF_CHECK_CUDA(cudaStreamWaitEvent(side->stream2, side->fork, 0));
      SPARF_CHECK_CUDA(cudaStreamWaitEvent(side->stream3, side->fork, 0));
      sd2 = side->stream2; sd3 = side->stream3;
    }

    // 3. weight-gradient jobs = (layer, slab of row tiles), one CTA on every SM but one, in a single wave.  A stage (32 rows of one tile) costs about the same ~2.4k clocks whatever its width (it is bound by
    //    the latency of the 3-deep HBM pipeline, profiles/r01_ncu_chain.md), so the slabs equalise the number of stages
    //    per CTA rather than bytes: 10 job types x ~14.8 slabs = 147 CTAs on a whole GPU.
    const int ctas = std::min(num_sms() - 1, kMaxWgradJobs);
    WgradJobs jobs;
    int nj = 0;
    auto add_jobs = [&](int tg, int tx, int mblk, int nblk, float* dW, int ldw, int col0, int enc, int slabs, float* colsum) {
      slabs = std::max(1, std::min(slabs, ntiles));
      for (int sl = 0; sl < slabs; ++sl, ++nj) {
        if (nj >= kMaxWgradJobs) continue;   // counted, rejected below
        WgradJob& j = jobs.j[nj];
        j.t_g = tg; j.t_x = tx; j.mblk = mblk; j.nblk = nblk;
        j.tile_begin = (int)((long long)ntiles * sl / slabs);
        j.tile_end = (int)((long long)ntiles * (sl + 1) / slabs);
        j.dW = dW; j.ldw = ldw; j.col0 = col0; j.enc_cols = enc; j.colsum = colsum;
        j.passes = wg_passes;
      }
    };
    int slabs[10];      // 8 wide job types, then the two encoder-block types
    const int s_lo = std::max(1, ctas / 10), extra = std::max(0, std::min(8, ctas - 10 * s_lo));
    for (int i = 0; i < 10; ++i) slabs[i] = s_lo + (i < extra ? 1 : 0);
    add_jobs(T_GHID, T_FEAT, 2, 4, grad->head_w[0], kW + kEv, 0, 0, slabs[7], grad->head_b[0]);     // head 0, feature part
    add_jobs(T_G7F, T_H0 + 6, 4, 4, grad->trunk_w[7] + kW, kW, 0, 0, slabs[0], grad->trunk_b[7] + 1);  // trunk 7 rows 1..256
    for (int l = 6; l >= 1; --l)
      add_jobs(t_g(l), T_H0 + (l - 1), 4, 4, grad->trunk_w[l], l == 4 ? kW + 63 : kW, 0, 0, slabs[7 - l], grad->trunk_b[l]);
    add_jobs(t_g(4), T_ENC, 4, 1, grad->trunk_w[4], kW + 63, kW, 1, slabs[8], nullptr);             // skip part of layer 4
    add_jobs(t_g(0), T_ENC, 4, 1, grad->trunk_w[0], 63, 0, 1, slabs[9], grad->trunk_b[0]);          // layer 0 (+ its bias)
    SPARF_REQUIRE(nj <= kMaxWgradJobs, "tc_mlp_backward: %d weight-gradient jobs exceed the table of %d", nj, kMaxWgradJobs);
    tc_mlp_wgrad_kernel<<<nj, 192, kWgSmem + 1024, st>>>(jobs, img);
    SPARF_CHECK_LAUNCH("tc_mlp_wgrad_kernel");

    // 4. CUDA-core leftovers: density row, 128->3 head, view-direction columns (bias gradients = column sums of the
    //    gradient images are produced inside the weight-gradient kernel)
    const int parts = (tape && wg_passes == 1) ? 1 : 2;     // forward images of a TC_3X_W1 tape hold their hi halves only
    const ReduceJob density{T_H0 + 6, 4, 1, c.g_raw, 1, grad->trunk_w[7], kW, grad->trunk_b[7], parts};   // density row of trunk 7
    const ReduceJob colour{T_HID, 2, 3, c.g_pre, 4, grad->head_w[1], kHW, grad->head_b[1], parts};         // 128 -> 3 colour layer
    const int tpb = 4;
    image_reduce_kernel<1><<<ceil_div(ntiles, tpb), 256, 0, sd>>>(density, img, Mc, ntiles, tpb);
    SPARF_CHECK_LAUNCH("image_reduce_kernel<1>");
    image_reduce_kernel<3><<<ceil_div(ntiles, tpb), 256, 0, sd2>>>(colour, img, Mc, ntiles, tpb);
    SPARF_CHECK_LAUNCH("image_reduce_kernel<3>");
    ray_sum_ghid_kernel<<<nr, 128, 0, sd2>>>(img, nr, S, c.rayS);
    SPARF_CHECK_LAUNCH("ray_sum_ghid_kernel");
    ray_head_wgrad_kernel<<<ceil_div(nr, 8), 128, 0, sd2>>>(nr, 8, c.rayS, c.denc, grad->head_w[0]);
    SPARF_CHECK_LAUNCH("ray_head_wgrad_kernel");

    // 5. gradients w.r.t. the rays (camera-pose optimisation)
    if (d_origins != nullptr || d_dirs != nullptr) {
      if (!tape) {
        pack_weights_enc_kernel<<<16, 256, 0, sd3>>>(mlp->trunk_w[4], mlp->trunk_w[0], c.packed_e);
        SPARF_CHECK_LAUNCH("pack_weights_enc_kernel");
      }
      EncGradParams ep;
      ep.packed = c.packed_e; ep.img = img; ep.t = t + m0;
      ep.d_origins = d_origins ? d_origins + (size_t)r0 * 3 : nullptr;
      ep.d_dirs = d_dirs ? d_dirs + (size_t)r0 * 3 : nullptr;
      ep.M = Mc; ep.S = S; ep.num_tiles = ntiles;
      tc_mlp_encgrad_kernel<<<std::min(ntiles, num_sms()), 192, kEgSmem + 1024, sd3>>>(ep);
      SPARF_CHECK_LAUNCH("tc_mlp_encgrad_kernel");
      if (d_dirs) {
        ray_head_dgrad_kernel<<<ceil_div(nr * 32, 256), 256, 0, sd2>>>(nr, c.rayS, mlp->head_w[0], c.gdenc);   // after ray_sum_ghid
        SPARF_CHECK_LAUNCH("ray_head_dgrad_kernel");
        if (sd3 != sd2) {   // direnc_bwd adds to d_dirs without atomics: after encgrad (same stream) and after gdenc is ready
          SPARF_CHECK_CUDA(cudaEventRecord(side->rayhead, sd2));
          SPARF_CHECK_CUDA(cudaStreamWaitEvent(sd3, side->rayhead, 0));
        }
        direnc_bwd_kernel<<<ceil_div(nr, 128), 128, 0, sd3>>>(nr, kLv, 32, c.denc, c.gdenc, dirs + (size_t)r0 * 3,
                                                             d_dirs + (size_t)r0 * 3);
        SPARF_CHECK_LAUNCH("direnc_bwd_kernel");
      }
    }
    // join: later work on the caller's stream (next chunk, optimiser, ...) sees every gradient
    SPARF_CHECK_CUDA(cudaEventRecord(side->join, side->stream));
    SPARF_CHECK_CUDA(cudaStreamWaitEvent(st, side->join, 0));
    if (sd2 != sd) {
      SPARF_CHECK_CUDA(cudaEventRecord(side->join2, sd2));
      SPARF_CHECK_CUDA(cudaStreamWaitEvent(st, side->join2, 0));
      SPARF_CHECK_CUDA(cudaEventRecord(side->join3, sd3));
      SPARF_CHECK_CUDA(cudaStreamWaitEvent(st, side->join3, 0));
    }
  }
  return SPARF_OK;
}

}  // namespace sparf
