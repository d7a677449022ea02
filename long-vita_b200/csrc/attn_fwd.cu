// Fused attention forward for sm_100a: softmax(scale * Q K^T + mask) V with online softmax, GQA,
// causal / zig-zag-causal / no mask, LSE output.
//
// One persistent CTA per SM, 12 warps, warp-specialised:
//   warp 0      TMA producer: Q tiles (2 x 128 rows per work item) and a K ring + V ring of
//               128-row tiles, 128-byte swizzle, mbarrier completion
//   warp 1      tcgen05.mma issuer (one elected thread).  S_t = Q_t K^T (SS form, both operands
//               from shared memory) into TMEM; O_t += P_t V (TS form: P read from TMEM, V from
//               shared memory as an MN-major operand).  Two query tiles are ping-ponged so the
//               tensor pipe works on tile 1-t while the softmax warps work on tile t:
//               QK0(j) PV1(j-1) QK1(j) PV0(j) ...
//   warps 2-3   idle in this kernel (the context-parallel variant uses them to pull remote K/V)
//   warps 4-7   softmax warpgroup for query tile 0 (one thread per query row)
//   warps 8-11  softmax warpgroup for query tile 1
// A softmax thread reads its row of S from TMEM (tcgen05.ld), keeps a running max in the log2
// domain, rescales O only when the max grew by more than 2^8 (lazy rescale: P <= 256 stays well
// inside bf16/fp32 range), writes P (bf16) back over S in TMEM (tcgen05.st) and at the end
// normalises O, stages it in the (now free) Q shared-memory tile and stores it with TMA.
//
// TMEM map (512 columns): S0/P0 @0, S1/P1 @128, O0 @256, O1 @256 + D.
//
// Reference call sites replaced: flash_attn_func / _flash_attention_forward in
// long_vita_megatron/core/transformer/dot_product_attention.py:318-326, 374-390 and
// long_vita/models/long_vita_qwen2_intern/flash_attention.py:52-74.
#include <cuda_bf16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace lv {

constexpr int A_BM = 128;   // query rows per tile
constexpr int A_BN = 128;   // key rows per tile
constexpr int A_THREADS = 384;

struct AttnKParams {
  int batch, sq, sk, hq, hkv;
  int causal;
  float scale_log2;
  int q_seg_len;
  long long q_seg_pos0, q_seg_pos1, kv_pos0;
  int n_qblk;      // ceil(sq / 256)
  int n_items;     // batch * hq * n_qblk
  int block_major; // 1: order work items (q-block, kv-head, head) - global longest-first; 0: (kv-head, q-block, head)
  int serpentine;  // 1: odd rounds sweep the item list backwards (default); LV_ATTN_SCHED=0 turns it off for A/B runs
  int poly_exp;    // 1: every 4th exponential of the softmax runs on the FMA pipe (polynomial), the rest on MUFU
  int mufu_turns;  // 1: the two softmax warps of an SM sub-partition take turns on its MUFU unit (LV_ATTN_TURNS=0: off)
  float* lse;
};

// Context-parallel extension (zig-zag layout, training/utils.py:329-341).  Every rank keeps its own
// K/V rows inside a peer-mapped ("symmetric") buffer; the copier warps of this kernel pull the
// chunks this rank's queries can see from the owning GPUs over NVLink into a local staging copy in
// global sequence order, 128-token block by block, and publish a per-block flag the TMA producer
// polls - so the K/V exchange is part of the attention kernel and overlaps its math.
struct CpKParams {
  int rank, cp;
  int chunk;                 // tokens per zig-zag chunk: S / (2 cp)
  int nblk_needed;           // 128-token key blocks this rank's queries can see
  uint32_t epoch1;           // epoch + 1 (flags are monotonic, never reset)
  int kv_row_elems;          // hkv * d
  long long peer_tok_stride; // elements between consecutive tokens in a peer's K|V rows
  const __nv_bfloat16* peer_kv[8];   // peer p: address of K of its local token 0 (V follows K in the row)
  uint32_t* peer_ready[8];           // peer p: its ready[parity][my rank] word
  const uint32_t* my_ready;          // ready[parity][0..cp)
  __nv_bfloat16* k_full;             // staging [S, hkv*d]
  __nv_bfloat16* v_full;
  uint32_t* blk_flags;               // [S / 128]
  uint32_t* fault;                   // sticky fault word (0 = healthy); set when a peer wait times out
  unsigned long long timeout_ns;     // bound of one wait on another GPU's progress
  unsigned long long order;          // chunk visiting order of this rank, 4 bits per entry (2 cp entries): its own two
                                     // chunks first, then the peers' by ring distance (rank - 1, rank - 2, ...)
  int tiles_per_chunk;               // chunk / 128
};

// Visiting order of the key tiles under context parallelism.  Online softmax does not care in which order the key
// tiles of a query row arrive, so every rank starts on the K/V rows it owns (no waiting at all) and then walks the
// peers in ring order - rank r reads from r-1 first, r-2 next ... - which staggers the ranks over the NVSwitch ports
// instead of all of them pulling chunk 0 from rank 0 at once (the "ring" schedule of TE / ring-flash-attn, SURVEY.md
// 8e).  The two query tiles of a work item share the K/V tiles, and tile t must take part in a PREFIX of the steps
// (steps j < n[t]): the tiles [0, lo) that both see come first, then [lo, hi), each range in chunk-priority order.
struct KvWalk {
  int lo, hi, a, b, li, g, gend;
  __device__ __forceinline__ void begin(int n0, int n1) {
    lo = min(n0, n1);
    hi = max(n0, n1);
    a = 0;
    b = lo;
    li = -1;
    g = gend = 0;
  }
  // global index of the next key tile (call exactly hi times per item)
  __device__ __forceinline__ int next(const CpKParams& c) {
    for (;;) {
      if (g < gend) return g++;
      if (++li >= 2 * c.cp) {       // first range done: the tiles only the longer query tile sees
        a = lo;
        b = hi;
        li = -1;
        continue;
      }
      const int ch = (int)((c.order >> (4 * li)) & 15ull);
      g = max(a, ch * c.tiles_per_chunk);
      gend = min(b, (ch + 1) * c.tiles_per_chunk);
    }
  }
};

// Waits on ANOTHER GPU's progress are bounded: a rank whose peer died (or never launched this layer) would otherwise
// spin forever and, because every other rank waits for it in turn, hang the whole node with no message.  After
// `timeout_ns` the waiter records a code in the sticky fault word and STOPS WAITING - the kernel finishes (its output
// is garbage), later waits of this and of the following launches return at once, and the host turns the word into
// LV_ESTATE at its next check (lv_cp_check_fault).  The clock is read every 1024 polls only.
constexpr uint32_t CP_FAULT_READY = 1u, CP_FAULT_BLOCK = 2u, CP_FAULT_EXIT = 4u;

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

struct PeerWait {
  unsigned long long t0 = 0;
  uint32_t polls = 0;
  // true: give up (fault already set by someone, or this wait timed out and sets it)
  __device__ __forceinline__ bool expired(const CpKParams& c, uint32_t code) {
    if ((++polls & 1023u) != 0) return false;
    if (*reinterpret_cast<volatile uint32_t*>(c.fault) != 0) return true;
    const unsigned long long now = global_ns();
    if (t0 == 0) {
      t0 = now;
      return false;
    }
    if (now - t0 > c.timeout_ns) {
      atomicOr(c.fault, code);
      return true;
    }
    return false;
  }
};

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_peer_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}

// 2^x on the FMA pipe (no MUFU): round-to-nearest split x = n + f, f in [-0.5, 0.5], cubic minimax for 2^f
// (max relative error 7.5e-5, tools/exp2_poly.py - 50x below the bf16 rounding P gets anyway), exponent
// add through the low mantissa bits of the magic-number sum.  x is clamped to >= -125 so the result
// stays a normal number: a masked -inf score becomes 2^-125 ~ 2e-38 instead of 0.  That is invisible in l and P V
// of a row with at least one visible key.  A row that sees no key at all would get l > 0 (2^-125 per polynomial
// exponential) and the mean of V, so the epilogues test a per-row flag (some visited tile had a finite maximum).
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -125.f);
  const float t = x + 12582912.f;            // 1.5 * 2^23: the integer part of x lands in the low mantissa bits
  const float f = x - (t - 12582912.f);
  float p = fmaf(0.055171321f, f, 0.24261054f);
  p = fmaf(p, f, 0.69326099f);
  p = fmaf(p, f, 0.99992811f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

// One 32-column chunk of a score row: P = 2^(S * scale_log2 - m), four partial row sums, bf16 pack.
// POLY: every 4th exponential is evaluated on the FMA pipe (ex2_poly), relieving the MUFU pipe that both
// softmax warpgroups share (16 ex2 / clk / SM = as many cycles as the two MMAs of a step at d = 128).
// Two exponentials at once on the FMA / ALU pipes with packed fp32 arithmetic (ex2_poly for a pair): 2 FMNMX (clamp),
// 3 FADD2 (magic-number split x = n + f), 3 FFMA2 (cubic), 2 LEA (exponent insert) = 5 issue slots per element and no
// MUFU slot, against 8 MUFU cycles per element otherwise.
__device__ __forceinline__ void ex2_poly_pair(float x0, float x1, float& p0, float& p1) {
  x0 = fmaxf(x0, -125.f);
  x1 = fmaxf(x1, -125.f);
  float t0, t1, n0, n1, f0, f1;
  fadd2(t0, t1, x0, x1, 12582912.f, 12582912.f);
  fadd2(n0, n1, t0, t1, -12582912.f, -12582912.f);
  fadd2(f0, f1, x0, x1, -n0, -n1);
  float q0, q1;
  ffma2v(q0, q1, f0, f1, 0.055171321f, 0.055171321f, 0.24261054f, 0.24261054f);
  ffma2v(q0, q1, q0, q1, f0, f1, 0.69326099f, 0.69326099f);
  ffma2v(q0, q1, q0, q1, f0, f1, 0.99992811f, 0.99992811f);
  p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(t0) << 23));
  p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(t1) << 23));
}

// One 32-column chunk of a score row: P = 2^(S * scale_log2 - m), four partial row sums, bf16 pack.
// POLY = number of element PAIRS per 8 (16 elements) whose exponentials run on the FMA pipe instead of the MUFU:
// 0 (none), 2 (25 %), 3 (37.5 %), 4 (50 %).  The MUFU unit delivers 4 results per cycle per SM sub-partition - a 128 x
// 128 tile keeps it busy 1024 cycles, as long as the tile's two MMAs - and is the softmax's bottleneck; the packed
// fp32 forms (2.5 issue slots per MUFU element, 6.5 per polynomial one) leave room to move part of the work over.
template <int POLY>
__device__ __forceinline__ void softmax_exp_chunk(const uint32_t (&sc)[32], float scale_log2, float neg_m, float& l0,
                                                  float& l1, float& l2, float& l3, uint32_t (&pk)[16]) {
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    float x0, x1, x2, x3;
    ffma2(x0, x1, __uint_as_float(sc[i + 0]), __uint_as_float(sc[i + 1]), scale_log2, neg_m);
    ffma2(x2, x3, __uint_as_float(sc[i + 2]), __uint_as_float(sc[i + 3]), scale_log2, neg_m);
    // pairs are numbered 0..7 inside a 16-element window; which of them take the polynomial is a compile-time pattern
    const int pair_a = (i / 2) & 7, pair_b = (i / 2 + 1) & 7;
    constexpr unsigned pattern = POLY == 2 ? 0x44u : (POLY == 3 ? 0x54u : (POLY == 4 ? 0xAAu : 0u));
    float p0, p1, p2, p3;
    if ((pattern >> pair_a) & 1u) {
      ex2_poly_pair(x0, x1, p0, p1);
    } else {
      p0 = ex2(x0);
      p1 = ex2(x1);
    }
    if ((pattern >> pair_b) & 1u) {
      ex2_poly_pair(x2, x3, p2, p3);
    } else {
      p2 = ex2(x2);
      p3 = ex2(x3);
    }
    fadd2(l0, l1, l0, l1, p0, p1);
    fadd2(l2, l3, l2, l3, p2, p3);
    pk[i / 2] = pack_bf16(p0, p1);
    pk[i / 2 + 1] = pack_bf16(p2, p3);
  }
}

// Exponentials on the FMA pipe, in element pairs per 8 pairs: LV_ATTN_POLY = 0 | 2 | 3 | 4 (default ATTN_POLY_DEFAULT).
constexpr int ATTN_POLY_DEFAULT = 2;   // measured round 2: 25 % is the best share at both head dims (profiles/README.md)
static int attn_poly_exp() {
  static const int v = [] {
    const char* e = getenv("LV_ATTN_POLY");
    if (e == nullptr) return ATTN_POLY_DEFAULT;
    const int x = atoi(e);
    return (x == 0 || x == 2 || x == 3 || x == 4) ? x : (x == 1 ? 2 : ATTN_POLY_DEFAULT);
  }();
  return v;
}

__device__ __forceinline__ void red_release_gpu_add(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Staging granularity: a 128-token key block is pulled as CP_SUB units of 32 tokens by different copier
// warps, and blk_flags[b] COUNTS completed units (it reaches CP_SUB * (epoch + 1) when block b of this
// epoch is whole).  With one unit per warp-visit and 8 x 16 B loads in flight per lane, a rank with few
// blocks (short sequences) still keeps every copier warp of the grid and ~1.2 MB of NVLink reads in
// flight; the first version moved one whole block per warp with 4 loads in flight and needed ~0.5 ms per
// layer at 18K tokens / 8 ranks, all of it exposed.
constexpr int CP_SUB = 4;
constexpr int CP_UNIT_ROWS = A_BN / CP_SUB;

__device__ __forceinline__ void cp_copier(const CpKParams& cpp, int warp, int lane) {
      const int cw = blockIdx.x * 2 + (warp - 2);          // copier index
      const int ncw = gridDim.x * 2;
      if (cw == 0) {
        // tell every peer that this rank's K/V rows for this epoch are complete (they were written
        // by earlier kernels on this stream; the fence orders them before the flag at system scope)
        __threadfence_system();
        if (lane < cpp.cp && lane != cpp.rank) st_release_sys(cpp.peer_ready[lane], cpp.epoch1);
      }
      uint32_t seen = 1u << cpp.rank;                      // peers whose ready flag has been observed
      const int vec_per_row = cpp.kv_row_elems / 4;        // 16-byte vectors in one K|V row pair
      const int vec_per_half = cpp.kv_row_elems / 8;
      const int n_units = cpp.nblk_needed * CP_SUB;
      for (int u = cw; u < n_units; u += ncw) {
        // the i-th block in this rank's chunk-priority order (own chunks, then peers by ring distance): the order in
        // which the query tiles consume them (KvWalk)
        int b = u / CP_SUB;
        {
          int i = b;
          for (int li = 0; li < 2 * cpp.cp; ++li) {
            const int ch = (int)((cpp.order >> (4 * li)) & 15ull);
            const int cnt = min(max(cpp.nblk_needed - ch * cpp.tiles_per_chunk, 0), cpp.tiles_per_chunk);
            if (i < cnt) {
              b = ch * cpp.tiles_per_chunk + i;
              break;
            }
            i -= cnt;
          }
        }
        const int tok0 = b * A_BN + (u % CP_SUB) * CP_UNIT_ROWS;
        const int chunk = tok0 / cpp.chunk;
        const int owner = chunk < cpp.cp ? chunk : 2 * cpp.cp - 1 - chunk;
        const int lrow0 = (chunk < cpp.cp ? 0 : cpp.chunk) + (tok0 - chunk * cpp.chunk);
        if (!(seen & (1u << owner))) {
          if (lane == 0)
            {
              [[maybe_unused]] uint32_t spins = 0;
              PeerWait pw;
              while (ld_acquire_sys(cpp.my_ready + owner) < cpp.epoch1) {
                LV_SPIN_GUARD(spins, "peer ready word", cpp.my_ready + owner, cpp.epoch1)
                if (pw.expired(cpp, CP_FAULT_READY)) break;
              }
            }
          __syncwarp();
          seen |= 1u << owner;
        }
        const __nv_bfloat16* src = cpp.peer_kv[owner] + (long long)lrow0 * cpp.peer_tok_stride;
        if (vec_per_row == 256) {
          // K|V row pair = 4 KB (8 kv heads x 128): one row per warp pass, 8 loads in flight per lane,
          // vectors 0..127 of the row are K, 128..255 are V
          const __nv_bfloat16* s_lane = src + lane * 8;
          __nv_bfloat16* dk = cpp.k_full + (long long)tok0 * cpp.kv_row_elems + lane * 8;
          __nv_bfloat16* dv = cpp.v_full + (long long)tok0 * cpp.kv_row_elems + lane * 8;
#pragma unroll 1
          for (int row = 0; row < CP_UNIT_ROWS; ++row) {
            uint4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = ld_peer_v4(s_lane + i * 256);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              *reinterpret_cast<uint4*>(dk + i * 256) = v[i];
              *reinterpret_cast<uint4*>(dv + i * 256) = v[4 + i];
            }
            s_lane += cpp.peer_tok_stride;
            dk += cpp.kv_row_elems;
            dv += cpp.kv_row_elems;
          }
        } else {
          const int total = CP_UNIT_ROWS * vec_per_row;
          for (int i0 = 0; i0 < total; i0 += 32 * 4) {
            uint4 v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k * 32 + lane;
              const int row = i / vec_per_row, col = i - row * vec_per_row;
              if (i < total) v[k] = ld_peer_v4(src + (long long)row * cpp.peer_tok_stride + col * 8);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = i0 + k * 32 + lane;
              const int row = i / vec_per_row, col = i - row * vec_per_row;
              if (i < total) {
                __nv_bfloat16* dst = col < vec_per_half
                                         ? cpp.k_full + (long long)(tok0 + row) * cpp.kv_row_elems + col * 8
                                         : cpp.v_full + (long long)(tok0 + row) * cpp.kv_row_elems + (col - vec_per_half) * 8;
                *reinterpret_cast<uint4*>(dst) = v[k];
              }
            }
          }
        }
        // the staged rows are read by TMA (async proxy): order this lane's generic-proxy stores before the
        // async proxy on the writer side as well (the producer fences again after its acquire)
        fence_proxy_async_all();
        __threadfence();
        __syncwarp();
        if (lane == 0) red_release_gpu_add(cpp.blk_flags + b, 1u);
      }
      if (cw == 0) {
        // do not retire before every peer has entered this epoch: a peer's flag for epoch e+1 then
        // proves it finished reading our epoch e-1 rows (buffer parity reuse, see DESIGN.md)
        if (lane < cpp.cp && lane != cpp.rank)
        {
          [[maybe_unused]] uint32_t spins = 0;
          PeerWait pw;
          while (ld_acquire_sys(cpp.my_ready + lane) < cpp.epoch1) {
            LV_SPIN_GUARD(spins, "peer epoch word (exit)", cpp.my_ready + lane, cpp.epoch1)
            if (pw.expired(cpp, CP_FAULT_EXIT)) break;
          }
        }
        __syncwarp();
      }
}

template <int D>
struct AttnCfg {
  static constexpr int KV_STAGES = (D == 128) ? 2 : 4;
  static constexpr int TILE_BYTES = 128 * D * 2;           // one 128-row tile of Q / K / V
  static constexpr int BOXES = D / 64;                     // 64-column (128-byte) TMA boxes per row
  // Q tiles of two work items in flight when they fit (head_dim 64: 4 x 16 KB): the next item's Q lands while this
  // one computes, and its first Q.K^T does not wait for this item's epilogue.  Short items - the ViT's 9 key tiles per
  // (frame, head, 256 rows) - otherwise pay an exposed TMA round trip (~1.5 us) per item.
  // (compile-time switch while the two-item path is being validated: -DLV_ATTN_QBUF64=2)
#ifndef LV_ATTN_QBUF64
#define LV_ATTN_QBUF64 1
#endif
  static constexpr int QBUF = (D == 64) ? LV_ATTN_QBUF64 : 1;
  static constexpr int SMEM_Q = QBUF * 2 * TILE_BYTES;
  static constexpr int SMEM_K = KV_STAGES * TILE_BYTES;
  static constexpr int SMEM_V = KV_STAGES * TILE_BYTES;
  static constexpr int SMEM_BAR = 512;
  static constexpr int SMEM_TOTAL = SMEM_Q + SMEM_K + SMEM_V + SMEM_BAR + 1024;
  static constexpr uint32_t TM_S0 = 0, TM_S1 = 128, TM_O0 = 256, TM_O1 = 256 + D;
};

// Static work assignment: the item list is sorted longest-first; CTAs sweep it boustrophedon (round r
// forwards, round r+1 backwards) so every CTA receives a near-equal share of causal work without a
// global atomic.  All warp roles of a CTA evaluate the same sequence.
__device__ __forceinline__ int sched_item(int round, int n_items, int serpentine) {
  const int base = round * (int)gridDim.x;
  if (base >= n_items) return -1;
  const int item = base + ((serpentine && (round & 1)) ? ((int)gridDim.x - 1 - (int)blockIdx.x) : (int)blockIdx.x);
  return item < n_items ? item : -1;
}

// (b, kv head, q-block rank, head-in-group) of a work item.  Head-major order keeps one kv head's K/V
// hot in L2 when all heads do not fit; block-major order is globally longest-first (better balance).
__device__ __forceinline__ void split_item(const AttnKParams& p, int item, int& b, int& kvh, int& rank, int& g) {
  const int G = p.hq / p.hkv;
  g = item % G;
  int r = item / G;
  if (p.block_major) {
    kvh = r % p.hkv;
    r /= p.hkv;
    rank = r % p.n_qblk;
    b = r / p.n_qblk;
  } else {
    rank = r % p.n_qblk;
    r /= p.n_qblk;
    kvh = r % p.hkv;
    b = r / p.hkv;
  }
}

struct WorkItem {
  int b, h, kvh, qblk;
  int n[2];          // kv tiles each query tile attends to (0: nothing to do)
  long long qpos[2]; // global position of row 0 of each query tile
  int row0[2];       // local row index of row 0 of each query tile
};

__device__ __forceinline__ WorkItem decode_item(const AttnKParams& p, int item) {
  WorkItem w;
  const int G = p.hq / p.hkv;
  int g, rank;
  split_item(p, item, w.b, w.kvh, rank, g);
  w.h = w.kvh * G + g;
  w.qblk = p.causal ? (p.n_qblk - 1 - rank) : rank;   // heaviest causal blocks first
  const int n_kv_tiles = (p.sk + A_BN - 1) / A_BN;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int row0 = w.qblk * 256 + t * A_BM;
    w.row0[t] = row0;
    const int seg = row0 / p.q_seg_len;
    w.qpos[t] = (seg == 0 ? p.q_seg_pos0 : p.q_seg_pos1) + (row0 - seg * p.q_seg_len);
    int n = 0;
    if (row0 < p.sq) {
      n = n_kv_tiles;
      if (p.causal) {
        const long long hi = w.qpos[t] + (A_BM - 1) - p.kv_pos0;  // last visible key index for the tile
        if (hi < 0)
          n = 0;
        else {
          const long long lim = hi / A_BN + 1;
          if (lim < n) n = (int)lim;
        }
      }
    }
    w.n[t] = n;
  }
  return w;
}

// POLY: every 4th exponential on the FMA pipe (ex2_poly).  TURNS: MUFU turn-taking of the two softmax warps of an
// SM sub-partition (see the softmax section).  Both are compile-time so the per-step loop carries no flag tests.
// HALF: the softmax warps publish P in two 64-key halves and the issuer starts the P.V k-steps of the first half while
// the exponentials of the second half are still running - it takes 256 of the 512 P.V cycles off the serial chain
// QK -> softmax -> PV of a query tile.
template <int D, bool CP, int POLY, bool TURNS, bool HALF>
__global__ void __launch_bounds__(A_THREADS, 1)
    attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                    const AttnKParams p, const CpKParams cpp) {
  using Cfg = AttnCfg<D>;
  constexpr int NS = Cfg::KV_STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::SMEM_Q;
  uint8_t* sV = sK + Cfg::SMEM_K;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + Cfg::SMEM_V);
  constexpr int QB = Cfg::QBUF;
  uint64_t* q_full = bars;            // [QB][2]
  uint64_t* q_empty = bars + 4;       // [QB][2]
  uint64_t* k_full = bars + 8;        // [NS]
  uint64_t* k_empty = bars + 8 + NS;  // [NS]
  uint64_t* v_full = bars + 8 + 2 * NS;
  uint64_t* v_empty = bars + 8 + 3 * NS;
  uint64_t* s_full = bars + 8 + 4 * NS;   // [2]
  uint64_t* p_full = s_full + 2;          // [2]
  uint64_t* o_full = p_full + 2;          // [2]
  uint64_t* o_free = o_full + 2;          // [2]: the epilogue has read O_t out of TMEM (the next item's first P.V overwrites it)
  uint64_t* tok = o_free + 2;             // [2 tiles][4 SM sub-partitions]: MUFU turn-taking, see the softmax warps
  uint64_t* p_half = tok + 8;             // [2]: the first 64 keys of P_t are in TMEM (HALF: P.V starts on them early)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_half + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 4; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_free[i], 4);
      mbar_init(&p_half[i], 4);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&tok[i], 1);
    for (int i = 0; i < NS; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    if (lane == 0) {
      uint32_t item_cnt = 0, kcnt = 0, vcnt = 0;
      KvWalk walk;
      for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
        const WorkItem w = decode_item(p, item);
        const int nmax = max(w.n[0], w.n[1]);
        if (CP) walk.begin(w.n[0], w.n[1]);
        const int qb = (int)(item_cnt % QB);
        const uint32_t qpar = (item_cnt / QB) & 1;
        auto load_kv = [&](int j) {
          int g = j;            // global key tile visited in step j
          if (CP) {
            g = walk.next(cpp);
            // staged by the copier warps of this GPU (any CTA)?  One L2 poll per tile; the K / V rings keep the
            // producer a step ahead of the tensor pipe, so the poll latency is off the critical path.
            {
              [[maybe_unused]] uint32_t spins = 0;
              PeerWait pw;
              while (ld_acquire_gpu(cpp.blk_flags + g) < cpp.epoch1 * CP_SUB) {
                LV_SPIN_GUARD(spins, "staged block flag", cpp.blk_flags + g, cpp.epoch1 * CP_SUB)
                if (pw.expired(cpp, CP_FAULT_BLOCK)) break;
              }
            }
            fence_proxy_async_all();   // copier warps wrote the staging rows through the generic proxy
          }
          {
            const int st = kcnt % NS;
            mbar_wait(&k_empty[st], ((kcnt / NS) & 1) ^ 1);
            mbar_arrive_expect_tx(&k_full[st], Cfg::TILE_BYTES);
            for (int bx = 0; bx < Cfg::BOXES; ++bx)
              tma_load_4d(sK + st * Cfg::TILE_BYTES + bx * 16384, &tmK, &k_full[st], bx * 64, g * A_BN, w.kvh, w.b,
                          kEvictLast);
            ++kcnt;
          }
          {
            const int st = vcnt % NS;
            mbar_wait(&v_empty[st], ((vcnt / NS) & 1) ^ 1);
            mbar_arrive_expect_tx(&v_full[st], Cfg::TILE_BYTES);
            for (int bx = 0; bx < Cfg::BOXES; ++bx)
              tma_load_4d(sV + st * Cfg::TILE_BYTES + bx * 16384, &tmV, &v_full[st], bx * 64, g * A_BN, w.kvh, w.b,
                          kEvictLast);
            ++vcnt;
          }
        };
        // With a single Q buffer the Q loads of this item wait for the previous item's epilogue; its first key tiles
        // do not (their ring slots free up as the previous item's last MMAs retire), so they are requested first.
        const int pre = (QB == 1) ? min(NS, nmax) : 0;
        for (int j = 0; j < pre; ++j) load_kv(j);
        for (int t = 0; t < 2; ++t) {
          mbar_wait(&q_empty[qb * 2 + t], qpar ^ 1);
          mbar_arrive_expect_tx(&q_full[qb * 2 + t], Cfg::TILE_BYTES);
          for (int bx = 0; bx < Cfg::BOXES; ++bx)
            tma_load_4d(sQ + (qb * 2 + t) * Cfg::TILE_BYTES + bx * 16384, &tmQ, &q_full[qb * 2 + t], bx * 64, w.row0[t], w.h, w.b,
                        kEvictFirst);
        }
        for (int j = pre; j < nmax; ++j) load_kv(j);
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    {
      // The whole warp executes this warp-uniform control flow and ONE elected lane issues the
      // tcgen05 instructions: descriptor arithmetic then lives in uniform registers.  (With the issue
      // loop under `if (lane == 0)` the compiler wrapped every MMA in an ELECT / R2UR.BROADCAST /
      // BRA.U.ANY sequence: ~73 issue cycles per 64-cycle MMA - the issuer was 64 % busy and bounded the
      // kernel, profiles/README.md.)
      constexpr uint32_t idesc_qk = make_idesc_bf16(A_BM, A_BN, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(A_BM, D, 0, 1);
      const uint32_t tS[2] = {tmem_base + Cfg::TM_S0, tmem_base + Cfg::TM_S1};
      const uint32_t tO[2] = {tmem_base + Cfg::TM_O0, tmem_base + Cfg::TM_O1};
      uint32_t item_cnt = 0, kcnt = 0, vcnt_wait = 0, vcnt_rel = 0;
      uint32_t pcnt[2] = {0, 0};
      uint32_t of_cnt[2] = {0, 0};     // items so far in which tile t had key tiles (= completed o_free[t] phases)

      // tiles are 1024-byte aligned, so stepping a descriptor is a plain add on its 14-bit address field
      const uint64_t qdesc0 = make_smem_desc(smem_u32(sQ), 16, 1024);
      uint64_t qdesc[2] = {qdesc0, qdesc0};
      const uint64_t kdesc0 = make_smem_desc(smem_u32(sK), 16, 1024);
      const uint64_t vdesc0 = make_smem_desc(smem_u32(sV), 16384, 1024);
      auto issue_qk = [&](int t, int kst) {
        const uint64_t qd = qdesc[t];
        const uint64_t kd = kdesc0 + (uint64_t)((kst * Cfg::TILE_BYTES) >> 4);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < D / 16; ++kk) {
            const uint32_t off = ((kk / 4) * 16384 + (kk % 4) * 32) >> 4;
            umma_ss(tS[t], qd + off, kd + off, idesc_qk, kk != 0 ? 1u : 0u);
          }
        }
        __syncwarp();
      };
      auto issue_pv = [&](int t, int vst, bool accumulate) {
        const uint64_t vd = vdesc0 + (uint64_t)((vst * Cfg::TILE_BYTES) >> 4);
        const bool leader = elect_one();
#pragma unroll
        for (int kk = 0; kk < A_BN / 16; ++kk) {
          if (HALF && kk == A_BN / 32) {
            // second half of P_t: pcnt[t] was advanced by the caller, so this step's phase is pcnt[t] - 1
            mbar_wait(&p_full[t], (pcnt[t] - 1) & 1);
            tc_fence_after();
          }
          // A: P_t rows in TMEM, 16 bf16 (= 8 columns) per k-step.  B: V tile, MN-major: 16 key rows
          // (2 KB) per k-step, the second 64 head-dim columns live one 16 KB box further.
          if (leader) umma_ts(tO[t], tS[t] + kk * 8, vd + (uint64_t)(kk * 128), idesc_pv, (accumulate || kk != 0) ? 1u : 0u);
        }
        __syncwarp();
      };
      auto commit = [&](uint64_t* bar) {
        if (elect_one()) umma_commit(bar);
        __syncwarp();
      };

      for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
        const WorkItem w = decode_item(p, item);
        const int n0 = w.n[0], n1 = w.n[1];
        const int nmax = max(n0, n1);
        const int qb = (int)(item_cnt % QB);
        const uint32_t qpar = (item_cnt / QB) & 1;
        qdesc[0] = qdesc0 + (uint64_t)(((qb * 2 + 0) * Cfg::TILE_BYTES) >> 4);
        qdesc[1] = qdesc0 + (uint64_t)(((qb * 2 + 1) * Cfg::TILE_BYTES) >> 4);
        mbar_wait(&q_full[qb * 2 + 0], qpar);
        mbar_wait(&q_full[qb * 2 + 1], qpar);
        tc_fence_after();
        // O_t of the previous item with key tiles read out by its epilogue?  o_free[t] completes one phase per item in
        // which tile t HAS key tiles (n[t] > 0) - both sides count those items the same way.  (Counting every item
        // let the epilogue warps of a tile without key tiles - the empty second tile of the ViT's last query block -
        // arrive for two consecutive items before the issuer looked: a parity wait cannot tell two phases from none.)
        bool o_waited[2] = {false, false};
        const uint32_t vbase = vcnt_wait;   // V tile j of this item has ring counter vbase + j
        for (int j = 0; j <= nmax; ++j) {
          int kst = 0;
          if (j < nmax) {
            kst = kcnt % NS;
            mbar_wait(&k_full[kst], (kcnt / NS) & 1);
            tc_fence_after();
          }
          if (j < n0) {
            issue_qk(0, kst);
            commit(&s_full[0]);
          }
          if (j >= 1) {
            if (j - 1 < n1) {
              const uint32_t vc = vbase + (j - 1);
              if (vc == vcnt_wait) {
                mbar_wait(&v_full[vc % NS], (vc / NS) & 1);
                ++vcnt_wait;
              }
              mbar_wait(HALF ? &p_half[1] : &p_full[1], pcnt[1] & 1);
              ++pcnt[1];
              if (!o_waited[1]) {
                if (of_cnt[1] > 0) mbar_wait(&o_free[1], (of_cnt[1] - 1) & 1);
                o_waited[1] = true;
              }
              tc_fence_after();
              issue_pv(1, vc % NS, j - 1 > 0);
              if (j - 1 == n1 - 1) commit(&o_full[1]);
            }
            // V(j-1) has now been consumed by every PV that needs it
            commit(&v_empty[vcnt_rel % NS]);
            ++vcnt_rel;
          }
          if (j < n1) {
            issue_qk(1, kst);
            commit(&s_full[1]);
          }
          if (j < nmax) {
            commit(&k_empty[kst]);
            ++kcnt;
          }
          if (j < n0) {
            const uint32_t vc = vbase + j;
            if (vc == vcnt_wait) {
              mbar_wait(&v_full[vc % NS], (vc / NS) & 1);
              ++vcnt_wait;
            }
            mbar_wait(HALF ? &p_half[0] : &p_full[0], pcnt[0] & 1);
            ++pcnt[0];
            if (!o_waited[0]) {
              if (of_cnt[0] > 0) mbar_wait(&o_free[0], (of_cnt[0] - 1) & 1);
              o_waited[0] = true;
            }
            tc_fence_after();
            issue_pv(0, vc % NS, j > 0);
            if (j == n0 - 1) commit(&o_full[0]);
          }
        }
        if (n0 > 0) ++of_cnt[0];
        if (n1 > 0) ++of_cnt[1];
      }
    }
  } else if (warp >= 4) {
    // =========================== softmax / epilogue warpgroups ===========================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    const int t = (warp - 4) >> 2;                // query tile handled by this warpgroup
    const int quad = warp & 3;                    // TMEM lane quadrant of this warp
    const int row = quad * 32 + lane;             // row inside the 128-row tile
    const int wg_tid = (warp - 4 - 4 * t) * 32 + lane;
    const uint32_t lane_base = uint32_t(quad * 32) << 16;
    const uint32_t tS = keep_u32(tmem_base + lane_base + (t == 0 ? Cfg::TM_S0 : Cfg::TM_S1));
    const uint32_t tO = keep_u32(tmem_base + lane_base + (t == 0 ? Cfg::TM_O0 : Cfg::TM_O1));
    uint32_t item_cnt = 0, scnt = 0, ocnt = 0;
    // Everything the per-step loop touches is resolved ONCE here: 32-bit shared-window addresses of its barriers
    // (a generic pointer costs an S2UR + uniform ALU chain per use), the scale, and per item the first step that
    // needs a mask.  The ncu source view of round 2 showed ~900 of the ~3800 cycles of a (2 x 128 rows) x 128 keys
    // step going to such scalar set-up on the softmax warps' critical path (profiles/README.md).
    const uint32_t a_sfull = keep_u32(smem_u32(&s_full[t])), a_pfull = keep_u32(smem_u32(&p_full[t]));
    const uint32_t a_ofull = keep_u32(smem_u32(&o_full[t])), a_ofree = keep_u32(smem_u32(&o_free[t]));
    const uint32_t a_phalf = keep_u32(smem_u32(&p_half[t]));
    // MUFU turn-taking (TURNS): the exponentials of one 128 x 128 score tile keep the MUFU unit of an SM sub-partition
    // busy for ~1050 cycles.  The two softmax warps of a sub-partition (one per query tile) take turns on it - tile
    // 0's warp runs exp(j), then tile 1's exp(j), then tile 0's exp(j+1) ... - so that the load / max / store /
    // hand-off parts of one warp overlap the exp phase of the other instead of both exp phases colliding.
    // tok[t][quad] is arrived by the OTHER tile's warp when its exp phase ends; waits and arrivals are paired exactly
    // (both sides know n[0], n[1] of the item).
    const uint32_t a_tok_mine = keep_u32(smem_u32(&tok[t * 4 + quad])), a_tok_other = keep_u32(smem_u32(&tok[(1 - t) * 4 + quad]));
    uint32_t tok_cnt = 0;
    const float scale_log2 = p.scale_log2;
    const int n_kv_tiles = (p.sk + A_BN - 1) / A_BN;
    const int j_ragged = (p.sk % A_BN) ? n_kv_tiles - 1 : 0x7fffffff;

    for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
      const WorkItem w = decode_item(p, item);
      const int n = w.n[t];
      const int n_other = w.n[1 - t];
      const int qb = (int)(item_cnt % QB);
      uint8_t* stage = sQ + (qb * 2 + t) * Cfg::TILE_BYTES;    // this item's Q_t tile doubles as the staging tile of O_t
      const long long qpos = w.qpos[t] + row;           // global position of this thread's query row
      // first key tile (GLOBAL index) that needs a mask: the diagonal ones (kv_pos0 + 128 g + 127 > position of the
      // tile's row 0) and the ragged last one
      KvWalk walk;
      if (CP) walk.begin(w.n[0], w.n[1]);
      int j_mask = j_ragged;
      if (p.causal) {
        const long long dd = w.qpos[t] - p.kv_pos0 - (A_BN - 1);
        const long long jd = dd < 0 ? 0 : dd / A_BN + 1;
        if (jd < j_mask) j_mask = (int)jd;
      }
      float m_used = 0.f, l = 0.f;
      bool seen = false;   // some visited tile holds a visible key of this row
      for (int j = 0; j < n; ++j) {
        int g = j;         // global key tile of this step (context parallelism visits them out of order)
        if (CP) g = walk.next(cpp);
        mbar_wait_a(a_sfull, scnt & 1);
        ++scnt;
        tc_fence_after();
        uint32_t s[128];
        tmem_ld128(tS, s);
        tmem_wait_ld();

        // ---- mask (only diagonal tiles and the ragged last key tile) ----
        // 32-column chunks with at least one visible key for some row of this warp (warp-uniform).  Only tracked at
        // head_dim 64 (the ViT's ragged 1025-key rows: 1 live chunk of 4 in every 9th tile); at head_dim 128 the test
        // per chunk costs more on every step than the skipped exponentials save on the rare diagonal tile.
        constexpr bool SKIP_DEAD = (D == 64);
        int live = 4;
        if (g >= j_mask) {
          const long long kidx0 = (long long)g * A_BN;
          long long lim = p.sk - kidx0;                               // first invalid column (ragged)
          long long lim_warp = lim;                                   // the same bound for the warp's LAST row
          if (p.causal) {
            const long long c = qpos - p.kv_pos0 - kidx0 + 1;         // first masked column (causal)
            if (c < lim) lim = c;
            const long long cw = c + (31 - lane);
            if (cw < lim_warp) lim_warp = cw;
          }
          const int ilim = lim < 0 ? 0 : (lim > A_BN ? A_BN : (int)lim);
#pragma unroll
          for (int i = 0; i < 128; ++i)
            if (i >= ilim) s[i] = 0xff800000u;  // -inf
          // chunks beyond the warp's last visible column hold only masked scores: their exponentials are skipped
          // (P = 0).  The ragged last key tile of the ViT (1025 = 8 x 128 + 1 keys) costs 1 chunk instead of 4.
          if (SKIP_DEAD) {
            const int lw = __shfl_sync(0xffffffffu, lim_warp < 0 ? 0 : (lim_warp > A_BN ? A_BN : (int)lim_warp), 0);
            live = (lw + 31) >> 5;
          }
        }

        // ---- row max: 8 independent chains ----
        float mx[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) mx[c] = fmax3(__uint_as_float(s[c * 16]), __uint_as_float(s[c * 16 + 1]), __uint_as_float(s[c * 16 + 2]));
#pragma unroll
        for (int c = 0; c < 8; ++c) {
#pragma unroll
          for (int i = 3; i < 15; i += 2) mx[c] = fmax3(mx[c], __uint_as_float(s[c * 16 + i]), __uint_as_float(s[c * 16 + i + 1]));
          mx[c] = fmaxf(mx[c], __uint_as_float(s[c * 16 + 15]));
        }
        const float mx_all = fmax3(fmax3(mx[0], mx[1], mx[2]), fmax3(mx[3], mx[4], mx[5]), fmaxf(mx[6], mx[7])) * scale_log2;
        seen |= mx_all > -INFINITY;

        // ---- lazy rescale ----
        if (j == 0) {
          m_used = (mx_all == -INFINITY) ? 0.f : mx_all;
        } else {
          const bool grow = mx_all > m_used + 8.f;
          if (__any_sync(0xffffffffu, grow)) {
            const float m_new = fmaxf(m_used, mx_all);
            const float alpha = ex2(m_used - m_new);
            m_used = m_new;
            l *= alpha;
#pragma unroll 1
            for (int c = 0; c < D / 32; ++c) {
              uint32_t o[32];
              tmem_ld32(tO + c * 32, o);
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
              tmem_st32(tO + c * 32, o);
            }
          }
        }

        // ---- P = exp2(S * scale_log2 - m), row sum, bf16 pack, store over S in TMEM ----
        const float neg_m = -m_used;
        float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
        if (TURNS) {
          // my turn on this sub-partition's MUFU?  tile 0 goes first in every step: it waits for tile 1's step j-1,
          // tile 1 waits for tile 0's step j (only where the other tile has that step at all)
          const bool need = (t == 0) ? (j >= 1 && j - 1 < n_other) : (j < n_other);
          if (need) {
            mbar_wait_a(a_tok_mine, tok_cnt & 1);
            ++tok_cnt;
          }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t pk[32];
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (!SKIP_DEAD || 2 * h + c < live) {
              softmax_exp_chunk<POLY>(reinterpret_cast<const uint32_t(&)[32]>(s[(2 * h + c) * 32]), scale_log2, neg_m, l0, l1, l2, l3,
                                      reinterpret_cast<uint32_t(&)[16]>(pk[c * 16]));
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) pk[c * 16 + i] = 0u;
            }
          }
          if (h == 1 && TURNS) {
            // the exponentials of this step are issued: hand the MUFU turn over (tile 0 -> tile 1's step j,
            // tile 1 -> tile 0's step j + 1) before the store / fence / hand-off tail of this step
            const bool give = (t == 0) ? (j < n_other) : (j + 1 < n_other);
            __syncwarp();
            if (give && lane == 0) mbar_arrive_a(a_tok_other);
          }
          tmem_st32(tS + h * 32, pk);
          if (HALF && h == 0) {
            tmem_wait_st();          // (also covers the lazy O rescale above)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_a(a_phalf);
          }
        }
        l += (l0 + l1) + (l2 + l3);
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_pfull);
      }

      // ---------------- epilogue: O / l -> bf16 -> smem (swizzled) -> TMA store; LSE ----------------
      const float inv_l = (seen && l > 0.f) ? 1.f / l : 0.f;
      if (n > 0) {
        mbar_wait_a(a_ofull, ocnt & 1);
        ++ocnt;
        tc_fence_after();
      } else {
        mbar_wait(&q_full[qb * 2 + t], (item_cnt / QB) & 1);   // the Q load into the staging tile must have landed
      }
#pragma unroll 1
      for (int c = 0; c < D / 32; ++c) {
        uint32_t o[32];
        if (n > 0) {
          tmem_ld32(tO + c * 32, o);
          tmem_wait_ld();
          if (c == D / 32 - 1) {
            // O_t is in registers: the next item's first P.V may overwrite the accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_a(a_ofree);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = 0u;
        }
        uint8_t* box = stage + (c >> 1) * 16384 + row * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 v;
          v.x = pack_bf16(__uint_as_float(o[8 * q + 0]) * inv_l, __uint_as_float(o[8 * q + 1]) * inv_l);
          v.y = pack_bf16(__uint_as_float(o[8 * q + 2]) * inv_l, __uint_as_float(o[8 * q + 3]) * inv_l);
          v.z = pack_bf16(__uint_as_float(o[8 * q + 4]) * inv_l, __uint_as_float(o[8 * q + 5]) * inv_l);
          v.w = pack_bf16(__uint_as_float(o[8 * q + 6]) * inv_l, __uint_as_float(o[8 * q + 7]) * inv_l);
          const int chunk = (c & 1) * 4 + q;
          *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v;
        }
      }
      tc_fence_before();
      if (p.lse != nullptr && w.row0[t] + row < p.sq) {
        const float lse = (seen && l > 0.f) ? (m_used + log2f(l)) * 0.69314718055994530942f : -INFINITY;
        p.lse[((long long)w.b * p.hq + w.h) * p.sq + w.row0[t] + row] = lse;
      }
      fence_proxy_async_smem();
      named_bar_sync(1 + t, 128);
      if (wg_tid == 0) {
        if (w.row0[t] < p.sq) {
          for (int bx = 0; bx < Cfg::BOXES; ++bx) tma_store_4d(&tmO, stage + bx * 16384, bx * 64, w.row0[t], w.h, w.b);
          tma_store_commit();
          tma_store_wait_read0();
        }
        mbar_arrive(&q_empty[qb * 2 + t]);   // this Q_t / staging tile may be overwritten by a later item's Q load
      }
    }
    if (wg_tid == 0) tma_store_wait_all0();
  } else {
    // =========================== warps 2-3: context-parallel K/V copier ===========================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
    if (CP) cp_copier(cpp, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// ================================================================================================
// Version 2 of the forward kernel: 64-key softmax steps with DOUBLE-BUFFERED S.
//
// v1 aliases P over the only S buffer of a query tile, so QK(j+1) cannot be issued before PV(j) and
// every iteration pays softmax latency + two mbarrier round trips on the tensor pipe's critical
// path (measured: 55 % tensor-pipe activity, softmax warps idle 47 % of the time waiting for S).
// Here each query tile owns two 64-column S buffers (TMEM: S0a S0b S1a S1b O0 O1 = 512 columns);
// the issuer runs one step ahead - QK_t(i+1) is queued before PV_t(i) - so S(i+1) is ready when
// softmax(i) retires and the chain becomes throughput- (MUFU / tensor) instead of latency-bound.
// Work per step and query tile: QK 128x64x128, PV 128x128x64.  Causal skipping is also 64-granular.
// ================================================================================================
constexpr int A_BH = 64;

struct WorkItem2 {
  int b, h, kvh;
  int n[2];           // 64-key steps per query tile
  long long qpos[2];
  int row0[2];
};

__device__ __forceinline__ WorkItem2 decode_item2(const AttnKParams& p, int item) {
  WorkItem2 w;
  const int G = p.hq / p.hkv;
  int g, rank;
  split_item(p, item, w.b, w.kvh, rank, g);
  w.h = w.kvh * G + g;
  const int qblk = p.causal ? (p.n_qblk - 1 - rank) : rank;
  const int n_steps = (p.sk + A_BH - 1) / A_BH;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int row0 = qblk * 256 + t * A_BM;
    w.row0[t] = row0;
    const int seg = row0 / p.q_seg_len;
    w.qpos[t] = (seg == 0 ? p.q_seg_pos0 : p.q_seg_pos1) + (row0 - seg * p.q_seg_len);
    int n = 0;
    if (row0 < p.sq) {
      n = n_steps;
      if (p.causal) {
        const long long hi = w.qpos[t] + (A_BM - 1) - p.kv_pos0;
        if (hi < 0)
          n = 0;
        else {
          const long long lim = hi / A_BH + 1;
          if (lim < n) n = (int)lim;
        }
      }
    }
    w.n[t] = n;
  }
  return w;
}

template <int D, bool CP>
__global__ void __launch_bounds__(A_THREADS, 1)
    attn_fwd2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                     const AttnKParams p, const CpKParams cpp) {
  using Cfg = AttnCfg<D>;
  constexpr int NS = Cfg::KV_STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::SMEM_Q;
  uint8_t* sV = sK + Cfg::SMEM_K;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + Cfg::SMEM_V);
  uint64_t* q_full = bars;            // [2]
  uint64_t* q_empty = bars + 2;       // [2]
  uint64_t* k_full = bars + 4;        // [NS]
  uint64_t* k_empty = bars + 4 + NS;
  uint64_t* v_full = bars + 4 + 2 * NS;
  uint64_t* v_empty = bars + 4 + 3 * NS;
  uint64_t* s_full = bars + 4 + 4 * NS;   // [2 tiles][2 buffers]
  uint64_t* p_full = s_full + 4;          // [2][2]
  uint64_t* o_done = p_full + 4;          // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
      mbar_init(&o_done[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
    }
    for (int i = 0; i < NS; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // TMEM columns: S_t[b] at t*128 + b*64; O_t at 256 + t*D

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      uint32_t item_cnt = 0, kcnt = 0, vcnt = 0;
      int ready_upto = 0;
      for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
        const WorkItem2 w = decode_item2(p, item);
        const int ntile = (max(w.n[0], w.n[1]) + 1) / 2;   // 128-row K/V tiles
        for (int t = 0; t < 2; ++t) {
          mbar_wait(&q_empty[t], (item_cnt & 1) ^ 1);
          mbar_arrive_expect_tx(&q_full[t], Cfg::TILE_BYTES);
          for (int bx = 0; bx < Cfg::BOXES; ++bx)
            tma_load_4d(sQ + t * Cfg::TILE_BYTES + bx * 16384, &tmQ, &q_full[t], bx * 64, w.row0[t], w.h, w.b,
                        kEvictFirst);
        }
        for (int j = 0; j < ntile; ++j) {
          if (CP && j >= ready_upto) {
            {
              [[maybe_unused]] uint32_t spins = 0;
              PeerWait pw;
              while (ld_acquire_gpu(cpp.blk_flags + j) < cpp.epoch1 * CP_SUB) {
                LV_SPIN_GUARD(spins, "staged block flag", cpp.blk_flags + j, cpp.epoch1 * CP_SUB)
                if (pw.expired(cpp, CP_FAULT_BLOCK)) break;
              }
            }
            ready_upto = j + 1;
            fence_proxy_async_all();
          }
          {
            const int st = kcnt % NS;
            mbar_wait(&k_empty[st], ((kcnt / NS) & 1) ^ 1);
            mbar_arrive_expect_tx(&k_full[st], Cfg::TILE_BYTES);
            for (int bx = 0; bx < Cfg::BOXES; ++bx)
              tma_load_4d(sK + st * Cfg::TILE_BYTES + bx * 16384, &tmK, &k_full[st], bx * 64, j * A_BN, w.kvh, w.b,
                          kEvictLast);
            ++kcnt;
          }
          {
            const int st = vcnt % NS;
            mbar_wait(&v_empty[st], ((vcnt / NS) & 1) ^ 1);
            mbar_arrive_expect_tx(&v_full[st], Cfg::TILE_BYTES);
            for (int bx = 0; bx < Cfg::BOXES; ++bx)
              tma_load_4d(sV + st * Cfg::TILE_BYTES + bx * 16384, &tmV, &v_full[st], bx * 64, j * A_BN, w.kvh, w.b,
                          kEvictLast);
            ++vcnt;
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    {   // warp-uniform control flow; one elected lane issues (see the v1 kernel)
      constexpr uint32_t idesc_qk = make_idesc_bf16(A_BM, A_BH, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(A_BM, D, 0, 1);
      uint32_t item_cnt = 0;
      uint32_t kbase = 0, vbase = 0;            // ring counters of this item's tile 0
      uint32_t scnt[2][2] = {{0, 0}, {0, 0}};   // completed uses of s_full / p_full [tile][buffer]
      for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
        const WorkItem2 w = decode_item2(p, item);
        const int nmax = max(w.n[0], w.n[1]);
        const int ntile = (nmax + 1) / 2;
        int k_waited = 0, v_waited = 0;
        mbar_wait(&q_full[0], item_cnt & 1);
        mbar_wait(&q_full[1], item_cnt & 1);
        tc_fence_after();

        auto issue_qk = [&](int t, int i) {
          const int m = i >> 1;
          while (k_waited <= m) {
            const uint32_t c = kbase + k_waited;
            mbar_wait(&k_full[c % NS], (c / NS) & 1);
            ++k_waited;
          }
          tc_fence_after();
          const int b = i & 1;
          const uint64_t qd = make_smem_desc(smem_u32(sQ + t * Cfg::TILE_BYTES), 16, 1024);
          const uint64_t kd = make_smem_desc(smem_u32(sK + ((kbase + m) % NS) * Cfg::TILE_BYTES) + (i & 1) * 8192, 16, 1024);
          const uint32_t d_tmem = tmem_base + t * 128 + b * 64;
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < D / 16; ++kk) {
              const uint32_t off = ((kk / 4) * 16384 + (kk % 4) * 32) >> 4;
              umma_ss(d_tmem, qd + off, kd + off, idesc_qk, kk != 0 ? 1u : 0u);
            }
            umma_commit(&s_full[t * 2 + b]);
          }
          __syncwarp();
        };
        auto issue_pv = [&](int t, int i) {
          const int m = i >> 1;
          while (v_waited <= m) {
            const uint32_t c = vbase + v_waited;
            mbar_wait(&v_full[c % NS], (c / NS) & 1);
            ++v_waited;
          }
          const int b = i & 1;
          mbar_wait(&p_full[t * 2 + b], scnt[t][b] & 1);
          ++scnt[t][b];
          tc_fence_after();
          const uint64_t vd = make_smem_desc(smem_u32(sV + ((vbase + m) % NS) * Cfg::TILE_BYTES) + (i & 1) * 8192, 16384, 1024);
          const uint32_t a_tmem = tmem_base + t * 128 + b * 64;
          const uint32_t d_tmem = tmem_base + 256 + t * D;
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < A_BH / 16; ++kk)
              umma_ts(d_tmem, a_tmem + kk * 8, vd + (uint64_t)(kk * 128), idesc_pv, (i > 0 || kk != 0) ? 1u : 0u);
            umma_commit(&o_done[t]);
          }
          __syncwarp();
        };

        for (int t = 0; t < 2; ++t)
          if (w.n[t] > 0) issue_qk(t, 0);
        auto commit = [&](uint64_t* bar) {
          if (elect_one()) umma_commit(bar);
          __syncwarp();
        };
        if (nmax == 1) commit(&k_empty[kbase % NS]);
        for (int i = 0; i < nmax; ++i) {
          const int s = i + 1;
          // queue the next step's QK^T of both tiles first (they need no softmax result), so the
          // tensor pipe has work while this step's probabilities are still being produced
          if (s < w.n[0]) issue_qk(0, s);
          if (s < w.n[1]) issue_qk(1, s);
          if (s < nmax && ((s & 1) == 1 || s == nmax - 1))
            commit(&k_empty[(kbase + (s >> 1)) % NS]);   // last QK on this K tile has been issued
          if (i < w.n[0]) issue_pv(0, i);
          if (i < w.n[1]) issue_pv(1, i);
          if ((i & 1) == 1 || i == nmax - 1) commit(&v_empty[(vbase + (i >> 1)) % NS]);
        }
        kbase += ntile;
        vbase += ntile;
      }
    }
  } else if (warp >= 4) {
    // =========================== softmax / epilogue warpgroups ===========================
    const int t = (warp - 4) >> 2;
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const int wg_tid = (warp - 4 - 4 * t) * 32 + lane;
    const uint32_t lane_base = uint32_t(quad * 32) << 16;
    const uint32_t tS = tmem_base + lane_base + t * 128;
    const uint32_t tO = tmem_base + lane_base + 256 + t * D;
    uint8_t* stage = sQ + t * Cfg::TILE_BYTES;
    uint32_t item_cnt = 0;
    uint32_t scnt[2] = {0, 0};   // uses of s_full[t][b]
    uint32_t pv_base = 0;        // PV commits on o_done[t] before this item

    for (int round = 0, item; (item = sched_item(round, p.n_items, p.serpentine)) >= 0; ++round, ++item_cnt) {
      const WorkItem2 w = decode_item2(p, item);
      const int n = w.n[t];
      const long long qpos = w.qpos[t] + row;
      float m_used = 0.f, l = 0.f;
      bool seen = false;   // some visited tile holds a visible key of this row
      for (int i = 0; i < n; ++i) {
        const int b = i & 1;
        mbar_wait(&s_full[t * 2 + b], scnt[b] & 1);
        ++scnt[b];
        tc_fence_after();
        uint32_t s[2][32];
        tmem_ld32(tS + b * 64, s[0]);
        tmem_ld32(tS + b * 64 + 32, s[1]);
        tmem_wait_ld();

        const long long kidx0 = (long long)i * A_BH;
        const bool ragged = kidx0 + A_BH > p.sk;
        const bool diag = p.causal && (p.kv_pos0 + kidx0 + A_BH - 1 > w.qpos[t]);
        if (ragged || diag) {
          long long lim = p.sk - kidx0;
          if (p.causal) {
            const long long c = qpos - p.kv_pos0 - kidx0 + 1;
            if (c < lim) lim = c;
          }
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int k = 0; k < 32; ++k)
              if (c * 32 + k >= lim) s[c][k] = 0xff800000u;
        }

        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int k = 0; k < 32; k += 4) {
          mx0 = fmax3(mx0, __uint_as_float(s[0][k]), __uint_as_float(s[0][k + 1]));
          mx1 = fmax3(mx1, __uint_as_float(s[0][k + 2]), __uint_as_float(s[0][k + 3]));
          mx2 = fmax3(mx2, __uint_as_float(s[1][k]), __uint_as_float(s[1][k + 1]));
          mx3 = fmax3(mx3, __uint_as_float(s[1][k + 2]), __uint_as_float(s[1][k + 3]));
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * p.scale_log2;
        seen |= mx > -INFINITY;

        float alpha = 1.f;
        bool rescale = false;
        if (i == 0) {
          m_used = (mx == -INFINITY) ? 0.f : mx;
        } else {
          const bool grow = mx > m_used + 8.f;
          rescale = __any_sync(0xffffffffu, grow);
          if (rescale) {
            const float m_new = fmaxf(m_used, mx);
            alpha = ex2(m_used - m_new);
            m_used = m_new;
            l *= alpha;
          }
        }

        const float neg_m = -m_used;
        float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t pk[16];
          if (p.poly_exp)
            softmax_exp_chunk<2>(s[c], p.scale_log2, neg_m, l0, l1, l2, l3, pk);
          else
            softmax_exp_chunk<0>(s[c], p.scale_log2, neg_m, l0, l1, l2, l3, pk);
          tmem_st16(tS + b * 64 + c * 16, pk);
        }
        l += (l0 + l1) + (l2 + l3);
        if (i > 0) {
          // PV_t(i-1) has normally retired long ago (QK_t(i) was queued before it, a whole softmax step
          // has passed).  Its phase is consumed here, every step and in order, so this thread can never
          // fall two phases behind o_done; O_t is rescaled (lazily) only after it.
          mbar_wait(&o_done[t], (pv_base + i - 1) & 1);
          if (rescale) {
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < D / 32; ++c) {
              uint32_t o[32];
              tmem_ld32(tO + c * 32, o);
              tmem_wait_ld();
#pragma unroll
              for (int k = 0; k < 32; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * alpha);
              tmem_st32(tO + c * 32, o);
            }
          }
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[t * 2 + b]);
      }

      // ---------------- epilogue ----------------
      const float inv_l = (seen && l > 0.f) ? 1.f / l : 0.f;
      if (n > 0) {
        mbar_wait(&o_done[t], (pv_base + n - 1) & 1);
        pv_base += n;
        tc_fence_after();
      } else {
        mbar_wait(&q_full[t], item_cnt & 1);
      }
#pragma unroll 1
      for (int c = 0; c < D / 32; ++c) {
        uint32_t o[32];
        if (n > 0) {
          tmem_ld32(tO + c * 32, o);
          tmem_wait_ld();
        } else {
#pragma unroll
          for (int k = 0; k < 32; ++k) o[k] = 0u;
        }
        uint8_t* box = stage + (c >> 1) * 16384 + row * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 v;
          v.x = pack_bf16(__uint_as_float(o[8 * q + 0]) * inv_l, __uint_as_float(o[8 * q + 1]) * inv_l);
          v.y = pack_bf16(__uint_as_float(o[8 * q + 2]) * inv_l, __uint_as_float(o[8 * q + 3]) * inv_l);
          v.z = pack_bf16(__uint_as_float(o[8 * q + 4]) * inv_l, __uint_as_float(o[8 * q + 5]) * inv_l);
          v.w = pack_bf16(__uint_as_float(o[8 * q + 6]) * inv_l, __uint_as_float(o[8 * q + 7]) * inv_l);
          const int chunk = (c & 1) * 4 + q;
          *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v;
        }
      }
      tc_fence_before();
      if (p.lse != nullptr && w.row0[t] + row < p.sq) {
        const float lse = (seen && l > 0.f) ? (m_used + log2f(l)) * 0.69314718055994530942f : -INFINITY;
        p.lse[((long long)w.b * p.hq + w.h) * p.sq + w.row0[t] + row] = lse;
      }
      fence_proxy_async_smem();
      named_bar_sync(1 + t, 128);
      if (wg_tid == 0) {
        if (w.row0[t] < p.sq) {
          for (int bx = 0; bx < Cfg::BOXES; ++bx) tma_store_4d(&tmO, stage + bx * 16384, bx * 64, w.row0[t], w.h, w.b);
          tma_store_commit();
          tma_store_wait_read0();
        }
        mbar_arrive(&q_empty[t]);
      }
    }
    if (wg_tid == 0) tma_store_wait_all0();
  } else {
    if (CP) cp_copier(cpp, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

template <int D, bool CP, int VER, int POLY = 0, bool TURNS = false, bool HALF = true>
static int launch_attn_t(const lv_attn_params* a, const CpKParams* cp, cudaStream_t s) {
  using Cfg = AttnCfg<D>;
  CUtensorMap tmQ, tmK, tmV, tmO;
  const uint32_t box[4] = {64, 128, 1, 1};
  {
    const uint64_t dims[4] = {(uint64_t)D, (uint64_t)a->sq, (uint64_t)a->hq, (uint64_t)a->batch};
    const uint64_t str[4] = {2, (uint64_t)a->q_strides[1] * 2, (uint64_t)a->q_strides[2] * 2, (uint64_t)a->q_strides[0] * 2};
    int r = encode_tmap_bf16(&tmQ, a->q, 4, dims, str, box, true);
    if (r) return r;
    const uint64_t ostr[4] = {2, (uint64_t)a->o_strides[1] * 2, (uint64_t)a->o_strides[2] * 2, (uint64_t)a->o_strides[0] * 2};
    r = encode_tmap_bf16(&tmO, a->out, 4, dims, ostr, box, true);
    if (r) return r;
  }
  {
    const uint64_t dims[4] = {(uint64_t)D, (uint64_t)a->sk, (uint64_t)a->hkv, (uint64_t)a->batch};
    const uint64_t kstr[4] = {2, (uint64_t)a->k_strides[1] * 2, (uint64_t)a->k_strides[2] * 2, (uint64_t)a->k_strides[0] * 2};
    const uint64_t vstr[4] = {2, (uint64_t)a->v_strides[1] * 2, (uint64_t)a->v_strides[2] * 2, (uint64_t)a->v_strides[0] * 2};
    int r = encode_tmap_bf16(&tmK, a->k, 4, dims, kstr, box, true);
    if (r) return r;
    r = encode_tmap_bf16(&tmV, a->v, 4, dims, vstr, box, true);
    if (r) return r;
  }
  AttnKParams p;
  p.batch = (int)a->batch;
  p.sq = (int)a->sq;
  p.sk = (int)a->sk;
  p.hq = (int)a->hq;
  p.hkv = (int)a->hkv;
  p.causal = a->causal ? 1 : 0;
  p.scale_log2 = a->scale * 1.4426950408889634f;
  p.q_seg_len = (int)a->q_seg_len;
  p.q_seg_pos0 = a->q_seg_pos[0];
  p.q_seg_pos1 = a->q_seg_pos[1];
  p.kv_pos0 = a->kv_pos0;
  p.n_qblk = (int)((a->sq + 255) / 256);
  p.n_items = (int)(a->batch * a->hq * p.n_qblk);
  // all kv heads' K and V fit comfortably in the 126 MB L2 -> global longest-first order
  p.block_major = (a->causal && a->sk * a->hkv * a->d * 4 <= (64ll << 20)) ? 1 : 0;
  static const int order_env = [] {   // LV_ATTN_ORDER=0 / 1 forces head-major / block-major order (A/B runs)
    const char* e = getenv("LV_ATTN_ORDER");
    return (e != nullptr && (e[0] == '0' || e[0] == '1')) ? (e[0] - '0') : -1;
  }();
  if (order_env >= 0 && a->causal) p.block_major = order_env;
  p.lse = a->lse;
  p.poly_exp = attn_poly_exp();      // read by the v2 kernel only (v1: template parameter)
  p.mufu_turns = TURNS ? 1 : 0;
  static const int serp = [] {
    const char* e = getenv("LV_ATTN_SCHED");
    return (e != nullptr && e[0] == '0') ? 0 : 1;
  }();
  p.serpentine = serp;
  static PerDeviceOnce attr_once;   // one per template instantiation
  int attr_dev;
  if (attr_once.needed(&attr_dev)) {
    if constexpr (VER == 2) {
      LV_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd2_kernel<D, CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_TOTAL));
    } else {
      LV_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<D, CP, POLY, TURNS, HALF>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_TOTAL));
    }
    attr_once.done(attr_dev);
  }
  int grid = p.n_items < sm_count() ? p.n_items : sm_count();
  CpKParams cpp;
  memset(&cpp, 0, sizeof(cpp));
  if (CP) {
    cpp = *cp;
    grid = sm_count();   // every copier warp takes part, also when there are fewer work items than SMs
  }
  if constexpr (VER == 2)
    attn_fwd2_kernel<D, CP><<<grid, A_THREADS, Cfg::SMEM_TOTAL, s>>>(tmQ, tmK, tmV, tmO, p, cpp);
  else
    attn_fwd_kernel<D, CP, POLY, TURNS, HALF><<<grid, A_THREADS, Cfg::SMEM_TOTAL, s>>>(tmQ, tmK, tmV, tmO, p, cpp);
  LV_CHECK_LAUNCH("attn_fwd_kernel");
  return LV_OK;
}

// LV_ATTN_TURNS=1 switches the MUFU turn-taking of the softmax warps on (default off: with two warps per sub-partition
// interleaving on the MUFU, 128K causal measured 1137 TFLOP/s without turns and 1076 with).  LV_ATTN_POLY=1: every
// 4th exponential on the FMA pipe.
static int attn_turns_env() {
  static const int v = [] {
    const char* e = getenv("LV_ATTN_TURNS");
    return (e != nullptr && (e[0] == '0' || e[0] == '1')) ? (e[0] - '0') : -1;
  }();
  return v;
}

template <int D, bool CP, int VER>
static int launch_attn(const lv_attn_params* a, const CpKParams* cp, cudaStream_t s) {
  if constexpr (VER == 2) {
    return launch_attn_t<D, CP, 2>(a, cp, s);
  } else {
    const bool turns = attn_turns_env() == 1;      // measured round 2: off is faster at both head dims (profiles/README.md)
    const int poly = attn_poly_exp();              // pairs per 8 on the FMA pipe: LV_ATTN_POLY = 0 | 2 | 3 | 4
    static const int half_env = [] {      // LV_ATTN_HALF=0: whole-tile P hand-off (A/B runs)
      const char* e = getenv("LV_ATTN_HALF");
      return (e != nullptr && e[0] == '0') ? 0 : 1;
    }();
    if constexpr (CP) {     // context-parallel launches: the default only (fewer instantiations of the big kernel)
      return launch_attn_t<D, CP, 1, ATTN_POLY_DEFAULT, false, true>(a, cp, s);
    } else {
      if (turns) return launch_attn_t<D, CP, 1, ATTN_POLY_DEFAULT, true, false>(a, cp, s);
      if (!half_env) return launch_attn_t<D, CP, 1, ATTN_POLY_DEFAULT, false, false>(a, cp, s);
      if (poly == 0) return launch_attn_t<D, CP, 1, 0, false, true>(a, cp, s);
      if (poly == 2) return launch_attn_t<D, CP, 1, 2, false, true>(a, cp, s);
      if (poly == 3) return launch_attn_t<D, CP, 1, 3, false, true>(a, cp, s);
      return launch_attn_t<D, CP, 1, 4, false, true>(a, cp, s);
    }
  }
}

}  // namespace lv

using namespace lv;

// LV_ATTN_VERSION: 1 = single-S-buffer kernel (default), 2 = double-buffered-S kernel (correct, slower).
static int attn_version() {
  static const int v = [] {
    const char* e = getenv("LV_ATTN_VERSION");
    return (e != nullptr && e[0] >= '1' && e[0] <= '2') ? (e[0] - '0') : 1;
  }();
  return v;
}

static int check_attn_params(const lv_attn_params* a) {
  LV_CHECK_ARG(a != nullptr, "lv_attn_fwd: null params");
  LV_CHECK_ARG(a->q && a->k && a->v && a->out, "lv_attn_fwd: null tensor pointer");
  LV_CHECK_ARG(a->d == 64 || a->d == 128, "lv_attn_fwd: head_dim %lld not supported (64, 128)", (long long)a->d);
  LV_CHECK_ARG(a->batch > 0 && a->sq > 0 && a->sk > 0 && a->hq > 0 && a->hkv > 0, "lv_attn_fwd: empty shape");
  LV_CHECK_ARG(a->hq % a->hkv == 0, "lv_attn_fwd: hq=%lld is not a multiple of hkv=%lld", (long long)a->hq, (long long)a->hkv);
  LV_CHECK_ARG(a->sq < (1ll << 30) && a->sk < (1ll << 30), "lv_attn_fwd: sequence too long");
  LV_CHECK_ARG(a->batch * a->hq * ((a->sq + 255) / 256) < (1ll << 31), "lv_attn_fwd: too many work items");
  LV_CHECK_ARG(a->q_seg_len > 0 && a->q_seg_len <= a->sq, "lv_attn_fwd: q_seg_len=%lld out of range", (long long)a->q_seg_len);
  if (a->q_seg_len < a->sq) {
    LV_CHECK_ARG(a->q_seg_len % 128 == 0 && a->sq <= 2 * a->q_seg_len, "lv_attn_fwd: segmented queries need q_seg_len %% 128 == 0 (a 128-row query tile never straddles segments) and at most two segments");
  }
  for (int i = 0; i < 3; ++i)
    LV_CHECK_ARG(a->q_strides[i] % 8 == 0 && a->k_strides[i] % 8 == 0 && a->v_strides[i] % 8 == 0 && a->o_strides[i] % 8 == 0,
                 "lv_attn_fwd: strides must be multiples of 8 elements (16 bytes)");
  return LV_OK;
}

extern "C" int lv_attn_fwd(const lv_attn_params* a, lv_stream_t stream) {
  int rc = check_attn_params(a);
  if (rc) return rc;
  LV_BIND_DEVICE(a->q);
  cudaStream_t s = (cudaStream_t)stream;
  // P is bf16 like V: tcgen05 kind::f16 faults on an fp16 A operand against a bf16 B operand
  // (measured on B200), so the fp16-P instantiation is never launched.
  if (attn_version() == 2) {
    if (a->d == 128) return launch_attn<128, false, 2>(a, nullptr, s);
    return launch_attn<64, false, 2>(a, nullptr, s);
  }
  if (a->d == 128) return launch_attn<128, false, 1>(a, nullptr, s);
  return launch_attn<64, false, 1>(a, nullptr, s);
}

extern "C" int lv_attn_cp_fwd(const lv_attn_params* a, const lv_cp_params* c, lv_stream_t stream) {
  int rc = check_attn_params(a);
  if (rc) return rc;
  LV_CHECK_ARG(c != nullptr, "lv_attn_cp_fwd: null cp params");
  LV_CHECK_ARG(c->cp >= 2 && c->cp <= 8 && c->rank >= 0 && c->rank < c->cp, "lv_attn_cp_fwd: bad rank %d / cp %d", c->rank, c->cp);
  LV_CHECK_ARG(a->batch == 1 && a->causal, "lv_attn_cp_fwd: batch 1, causal only");
  LV_CHECK_ARG(a->d == 128, "lv_attn_cp_fwd: head_dim 128 only");
  const int64_t S = c->seq_total;
  LV_CHECK_ARG(S % (2 * c->cp) == 0, "lv_attn_cp_fwd: seq_total %lld not divisible by 2*cp", (long long)S);
  const int64_t chunk = S / (2 * c->cp);
  LV_CHECK_ARG(chunk % 128 == 0, "lv_attn_cp_fwd: chunk %lld must be a multiple of 128 tokens", (long long)chunk);
  LV_CHECK_ARG(a->sq == 2 * chunk && a->sk == S && a->q_seg_len == chunk && a->kv_pos0 == 0,
               "lv_attn_cp_fwd: expects sq = 2*chunk local queries against the S-row staging buffers");
  LV_CHECK_ARG(a->q_seg_pos[0] == c->rank * chunk && a->q_seg_pos[1] == (2 * c->cp - 1 - c->rank) * chunk,
               "lv_attn_cp_fwd: q_seg_pos does not match the zig-zag layout of rank %d", c->rank);
  LV_CHECK_ARG(a->k == c->k_full && a->v == c->v_full, "lv_attn_cp_fwd: k / v must be the staging buffers");
  LV_CHECK_ARG(c->my_ready && c->blk_flags && c->k_full && c->v_full, "lv_attn_cp_fwd: null cp buffer");
  CpKParams k;
  memset(&k, 0, sizeof(k));
  k.rank = c->rank;
  k.cp = c->cp;
  k.chunk = (int)chunk;
  k.nblk_needed = (int)((2 * c->cp - c->rank) * chunk / A_BN);
  k.epoch1 = c->epoch + 1;
  k.kv_row_elems = (int)(a->hkv * a->d);
  k.peer_tok_stride = c->peer_tok_stride;
  const int parity = (int)(c->epoch & 1);
  for (int p = 0; p < c->cp; ++p) {
    LV_CHECK_ARG(c->peer_kv[p] != nullptr && c->peer_ready[p] != nullptr, "lv_attn_cp_fwd: null peer pointer for rank %d", p);
    k.peer_kv[p] = reinterpret_cast<const __nv_bfloat16*>(c->peer_kv[p]);
    k.peer_ready[p] = reinterpret_cast<uint32_t*>(c->peer_ready[p]) + parity * 8 + c->rank;
  }
  LV_BIND_DEVICE(a->q);     // after every argument check, so that bad arguments are reported without touching CUDA
  k.my_ready = reinterpret_cast<const uint32_t*>(c->my_ready) + parity * 8;
  k.k_full = reinterpret_cast<__nv_bfloat16*>(c->k_full);
  k.v_full = reinterpret_cast<__nv_bfloat16*>(c->v_full);
  k.blk_flags = reinterpret_cast<uint32_t*>(c->blk_flags);
  LV_CHECK_ARG(c->fault != nullptr, "lv_attn_cp_fwd: null fault word");
  k.fault = reinterpret_cast<uint32_t*>(c->fault);
  static const unsigned long long timeout_ms = [] {
    const char* e = getenv("LV_CP_TIMEOUT_MS");
    const long long v = e ? atoll(e) : 0;
    return (unsigned long long)(v > 0 ? v : 120000);      // 2 minutes: far beyond any rank skew of a healthy job
  }();
  k.timeout_ns = timeout_ms * 1000000ull;
  // Chunk visiting order.  Default: plain global order - the result is then BIT-IDENTICAL to the single-device kernel
  // on the gathered K/V (same key order, same rounding sequence), which is what bench.py's in-run parity check
  // asserts.  LV_CP_ORDER=1: own chunks first, then the peers' by ring distance; measured on 8 GPUs at 18K tokens:
  // 107.46 ms per prefill against 107.48 ms in global order (the exchange is not what bounds that configuration), and
  // the output then differs from the single-device kernel by the rounding of a different summation order (3.1e-3
  // relative between the two bf16 results; both within the test bound against the fp32 oracle).
  k.tiles_per_chunk = (int)(chunk / A_BN);
  static const int ring_order = [] {
    const char* e = getenv("LV_CP_ORDER");
    return (e != nullptr && e[0] == '1') ? 1 : 0;
  }();
  k.order = 0;
  for (int i = 0; i < c->cp; ++i) {
    const int peer = ring_order ? (c->rank - i + c->cp) % c->cp : i;
    const unsigned long long first = ring_order ? (unsigned long long)peer : (unsigned long long)(2 * i);
    const unsigned long long second = ring_order ? (unsigned long long)(2 * c->cp - 1 - peer) : (unsigned long long)(2 * i + 1);
    k.order |= first << (4 * (2 * i));
    k.order |= second << (4 * (2 * i + 1));
  }
  if (attn_version() == 2) return launch_attn<128, true, 2>(a, &k, (cudaStream_t)stream);
  return launch_attn<128, true, 1>(a, &k, (cudaStream_t)stream);
}

// Peer-mappable ("symmetric") allocations for the context-parallel K/V exchange: plain cudaMalloc
// memory exported / imported with CUDA IPC handles (64 opaque bytes the host exchanges over
// torch.distributed).
extern "C" int lv_ipc_alloc(int64_t bytes, void** ptr) {
  LV_CHECK_ARG(ptr != nullptr && bytes > 0, "lv_ipc_alloc: bad arguments");
  LV_CHECK_CUDA(cudaMalloc(ptr, (size_t)bytes));
  LV_CHECK_CUDA(cudaMemset(*ptr, 0, (size_t)bytes));
  return LV_OK;
}
extern "C" int lv_ipc_free(void* ptr) {
  if (ptr) LV_CHECK_CUDA(cudaFree(ptr));
  return LV_OK;
}
extern "C" int lv_ipc_get_handle(void* ptr, void* handle64) {
  LV_CHECK_ARG(ptr && handle64, "lv_ipc_get_handle: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  LV_CHECK_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle64, &h, 64);
  return LV_OK;
}
extern "C" int lv_ipc_open_handle(const void* handle64, void** ptr) {
  LV_CHECK_ARG(ptr && handle64, "lv_ipc_open_handle: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  LV_CHECK_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return LV_OK;
}
// Read (and keep) the sticky fault word of a context-parallel context: LV_OK when healthy, LV_ESTATE with a message
// naming what timed out otherwise.  Synchronises `stream` (the word is written by kernels on it).
extern "C" int lv_cp_check_fault(const void* fault, lv_stream_t stream) {
  LV_CHECK_ARG(fault != nullptr, "lv_cp_check_fault: null pointer");
  LV_BIND_DEVICE(fault);
  uint32_t w = 0;
  LV_CHECK_CUDA(cudaMemcpyAsync(&w, fault, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  LV_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (w == 0) return LV_OK;
  lv::set_error("context-parallel exchange timed out (fault word 0x%x:%s%s%s): a peer rank did not publish its K/V rows "
                "for this layer in time - it died, hung, or is not running the same sequence of attention calls",
                w, (w & CP_FAULT_READY) ? " peer-ready" : "", (w & CP_FAULT_BLOCK) ? " staged-block" : "",
                (w & CP_FAULT_EXIT) ? " exit-handshake" : "");
  return LV_ESTATE;
}

extern "C" int lv_ipc_close_handle(void* ptr) {
  if (ptr) LV_CHECK_CUDA(cudaIpcCloseMemHandle(ptr));
  return LV_OK;
}
