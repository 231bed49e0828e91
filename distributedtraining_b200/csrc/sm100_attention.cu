// Causal self-attention for sm_100a on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands by TMA).
//
// Layout: packed qkv [M = B*T, (H + 2*Hkv) * hd] bf16 (q heads | k heads | v heads), head_dim hd in {64, 128}: every kernel
// is a template over HD.  An operand tile [128 rows x HD] is HD / 64 consecutive 128B-swizzle atoms [128 x 64] (16 KB each),
// loaded as HD / 64 TMA boxes; K-major products over hd step (k >> 2) atoms + (k & 3) * 32 B, MN-major operands with N = HD
// use LBO = atom stride (the same addressing as the two-atom P tile).
// Tokens are treated as ONE flat axis of M rows cut into 128-row blocks; the mask is
//        valid(r, c)  <=>  seq_start(r) <= c <= r            (same sequence AND causal)
// so short sequences (the reference miner trains on T = 64: reference neurons/miner.py:70) are packed two per tile and
// long ones (T = 512 validator/averager batches: neurons/validator.py:63) loop over KV blocks with online softmax.
//
// forward   (grid: q-block x head):    S = Q K^T -> softmax (fp32, exp2) -> P (bf16, smem) -> O += P V
// backward  (two kernels, no atomics): KV-owner CTA accumulates dK, dV in TMEM over all q-blocks (and the q heads of
//                                      its GQA group); Q-owner CTA accumulates dQ in TMEM over its kv-blocks.
// P / dS tiles are written once to shared memory in the 128B-swizzled layout that is simultaneously a valid K-major
// A operand (P V, dS K) and a valid MN-major A operand (P^T dO, dS^T Q) -- no transposes anywhere.
//
// Parity: replaces HF GPT-2's eager/SDPA attention inside the reference's model(...) / loss.backward()
// (reference hivetrain/training_manager.py:380-386; SURVEY.md K4, K9).
#include <cstdint>
#include <cstdlib>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "dropout.cuh"
#include "launch_pdl.cuh"
#include "sm100_ptx.cuh"

namespace dtb {

int make_tmap_2d(CUtensorMap* out, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t pitch_elems,
                 uint32_t box_inner, uint32_t box_outer);  // sm100_gemm.cu

constexpr int kBlk = 128;        // token rows per block (q and kv)
constexpr int kTile = kBlk * 64 * 2;  // 16 KB: one [128 x 64] bf16 128B-swizzle atom (a head-dim-64 tile, half of a 128 one)
constexpr int kSmemLimit = 232448;     // 227 KB of dynamic shared memory per block
constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
  CUtensorMap tmap_qkv;  // [M, qkv_dim], box 64 x 128
  CUtensorMap tmap_do;   // [M, H*hd],   box 64 x 128 (backward)
  CUtensorMap tmap_o;    // [M, H*hd],   box 64 x 128 (backward, single-block kernel: O tile for D = rowsum(dO * O))
  CUtensorMap tmap_out;  // forward: out [M, H*hd]; backward: dqkv [M, qkv_dim]; box 64 x 128 (single-block kernels store by TMA)
  const __nv_bfloat16* o;
  const __nv_bfloat16* dout;
  __nv_bfloat16* out;    // forward output / backward dqkv
  float* lse;            // [B, H, T]
  int M, T, H, Hkv, ld_out, ld_o;
  float scale;
  const int* kv_len;     // optional [B]: keys >= seq_start + kv_len[b] are masked for EVERY query row of sequence b (HF attention_mask
                         // of a right-padded batch: reference hivetrain/training_manager.py:380-384); nullptr = causal only
  float* dbias;          // backward, single-block kernel only: += column sums of dqkv (the qkv bias gradient), fp32 [qkv_dim]
  DropArgs drop;  // attention-probability dropout (GPT-2 attn_pdrop): P is masked AFTER the softmax normaliser is formed
};

// multiply 32 consecutive probabilities (key tokens kg0 .. kg0+31, kg0 even) of one (head, q row) by their dropout factors
DTB_DEVICE void drop_p32(float* s, uint32_t rowkey, int kg0, uint32_t thr, float scale) {
  const uint32_t pair0 = uint32_t(kg0) >> 1;
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    const uint32_t w = drop_word(rowkey, pair0 + (i >> 1));
    s[i] *= drop_mul_lo(w, thr, scale);
    s[i + 1] *= drop_mul_hi(w, thr, scale);
  }
}
DTB_DEVICE uint32_t attn_row_key(const AttnParams& p, int h, int row_tok) {
  return p.drop.thr ? drop_row_key(drop_key(p.drop.rng, p.drop.stream), uint32_t(h) * uint32_t(p.M) + uint32_t(row_tok)) : 0u;
}

// last valid key token (absolute index) of query row `row_tok`: causal AND inside the un-padded prefix of its sequence
DTB_DEVICE int row_last_key(const AttnParams& p, int row_tok) {
  if (row_tok >= p.M) return -1;
  int hi = row_tok;
  if (p.kv_len) {
    const int b = row_tok / p.T;
    hi = min(hi, b * p.T + max(p.kv_len[b], 1) - 1);
  }
  return hi;
}

DTB_DEVICE uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
DTB_DEVICE void tmem_ld32(uint32_t taddr, float* f) {
  uint32_t r[32];
  tmem_ld_32x32b_x32(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(r[i]);
}
DTB_DEVICE void tmem_ld32x2(uint32_t ta, float* a, uint32_t tb, float* b) {
  uint32_t ra[32], rb[32];
  tmem_ld_32x32b_x32(ta, ra);
  tmem_ld_32x32b_x32(tb, rb);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    a[i] = __uint_as_float(ra[i]);
    b[i] = __uint_as_float(rb[i]);
  }
}
// write 8 bf16 (16 B) of row `row`, logical 16B-chunk `ch` (0..7) into a [128 x 128 B] 128B-swizzled tile
DTB_DEVICE void st_swz(uint8_t* tile, int row, int ch, uint4 v) {
  *reinterpret_cast<uint4*>(tile + row * 128 + ((ch ^ (row & 7)) << 4)) = v;
}
// one [128 x HD] operand tile = HD / 64 TMA boxes (atoms) at columns col, col + 64, ...
template <int HD>
DTB_DEVICE void tma_load_tile(uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int col, int row) {
#pragma unroll
  for (int a = 0; a < HD / 64; ++a) tma_load_2d(dst + a * kTile, map, bar, col + a * 64, row);
}
template <int HD>
DTB_DEVICE void tma_store_tile(const CUtensorMap* map, uint8_t* src, int col, int row) {
#pragma unroll
  for (int a = 0; a < HD / 64; ++a) tma_store_2d(map, src + a * kTile, col + a * 64, row);
}
// descriptor offset (16 B units) of K-step k (16 bf16 = 32 B) of a K-major operand whose K extent spans 64-column atoms
DTB_DEVICE constexpr uint64_t kstep_off(int k) { return uint64_t((k >> 2) * (kTile >> 4) + (k & 3) * 2); }

// ---- softmax building blocks (one thread = one query row, 32-column chunks read from TMEM) -------------------------
// ncu of the T = 512 kernels (profiles/ncu_r2_attn_tiled.md): 27 SASS instructions per score, 25 % issue utilisation at 2 warps
// per scheduler -- per-element mask compares, the denormal-safe exp2f() expansion and serial max / sum chains.  Hence:
// MUFU.EX2 directly, the mask as one 32-bit word per chunk (warp-uniform all / none fast paths), four independent chains.
DTB_DEVICE float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// bit i set  <=>  column ch * 32 + i is a valid key for this row (c_lo <= c <= c_hi)
DTB_DEVICE uint32_t chunk_mask(int c_lo, int c_hi, int ch) {
  const int lo = max(c_lo - ch * 32, 0), hi = min(c_hi - ch * 32, 31);
  return lo > hi ? 0u : ((0xffffffffu >> (31 - hi)) & (0xffffffffu << lo));
}
template <bool MASKED>
DTB_DEVICE float chunk_rowmax(const float* s, uint32_t vm) {
  float m[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
  for (int i = 0; i < 32; ++i) m[i & 3] = fmaxf(m[i & 3], (!MASKED || ((vm >> i) & 1u)) ? s[i] : -CUDART_INF_F);
  return fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
}
// s[i] <- 2^(s[i] * sl2 - mref) (0 where masked); returns the chunk's sum
template <bool MASKED>
DTB_DEVICE float chunk_exp(float* s, uint32_t vm, float sl2, float mref) {
  float l[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    float e = ex2_fast(fmaf(s[i], sl2, -mref));
    if (MASKED) e = ((vm >> i) & 1u) ? e : 0.f;
    s[i] = e;
    l[i & 3] += e;
  }
  return (l[0] + l[1]) + (l[2] + l[3]);
}
// Longest-first CTA order for the tiled kernels.  Causal cost grows with the block's position inside its sequence (q-owner
// CTAs: position + 1 kv blocks; kv-owner CTAs: blocks-per-sequence - position q blocks), and the grid is 1.3 - 2.6 waves, so
// in natural order a 4-iteration CTA that starts in the tail sets the kernel time.  Linear CTA id (= dispatch order) ->
// (block, head) with all heaviest blocks first.  Identity unless the batch is whole sequences of a multiple of 128 tokens.
DTB_DEVICE void lpt_block(const AttnParams& p, bool heavy_last, int& blk, int& h) {
  blk = blockIdx.x;
  h = blockIdx.y;
  const int nps = p.T / kBlk;
  if (nps <= 1 || p.T % kBlk != 0 || p.M % p.T != 0) return;
  const int heads = gridDim.y, per_class = (p.M / p.T) * heads;
  const int L = blockIdx.y * gridDim.x + blockIdx.x;
  const int cls = L / per_class, idx = L - cls * per_class;  // cls 0 = heaviest
  h = idx % heads;
  blk = (idx / heads) * nps + (heavy_last ? nps - 1 - cls : cls);
}

constexpr uint32_t kFullWarp = 0xffffffffu;

// ------------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------------
// smem: Q | K0 V0 | K1 V1 | P(2 atoms)   hd 64: 16 + 64 + 32 = 112 KB -> 2 CTAs / SM;  hd 128: 32 + 128 + 32 = 192 KB -> 1
// TMEM: S[128] | O[hd] -> 256 columns.  The output row is accumulated in registers (acc[HD]).
template <int HD>
constexpr int fwd_smem() { return 1024 + kTile * (5 * (HD / 64) + 2) + 64; }
static_assert(fwd_smem<64>() <= kSmemLimit / 2 && fwd_smem<128>() <= kSmemLimit, "attn_fwd smem budget");

template <int HD>
__global__ void __launch_bounds__(128, HD == 64 ? 2 : 1) attn_fwd_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kOp = kTile * (HD / 64);  // one [128 x HD] operand tile
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // PDL: a dependent GEMM may start its prologue (sm100_ptx.cuh)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + kOp;         // [2 stages][K, V]
  uint8_t* sP = smem + kOp * 5;      // 2 atoms (keys 0-63 | 64-127)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOp * 5 + 2 * kTile);
  uint64_t* bar_q = bars;            // Q landed
  uint64_t* bar_kv = bars + 1;       // [2] K/V stage landed
  uint64_t* bar_s = bars + 3;        // S ready
  uint64_t* bar_o = bars + 4;        // P V done
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x, warp = tid >> 5;
  int qb, h;
  lpt_block(p, true, qb, h);
  const int hk = h / (p.H / p.Hkv);
  const int q0 = qb * kBlk;
  const int row_tok = q0 + tid;
  const int seq_start = (row_tok / p.T) * p.T;
  const int kb_first = ((q0 / p.T) * p.T) / kBlk;  // kv block holding the start of the first row's sequence
  const int nkb = qb - kb_first + 1;
  const int colQ = h * HD, colK = (p.H + hk) * HD, colV = (p.H + p.Hkv + hk) * HD;

  if (tid == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    mbar_init(bar_q, 1);
    mbar_init(&bar_kv[0], 1);
    mbar_init(&bar_kv[1], 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_o, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  const uint32_t tS = tmem, tO = tmem + 128;
  const uint32_t lane_off = (uint32_t(warp) * 32u) << 16;

  if (tid == 0) {
    mbar_expect_tx(bar_q, kOp);
    tma_load_tile<HD>(sQ, &p.tmap_qkv, bar_q, colQ, q0);
    mbar_expect_tx(&bar_kv[0], 2 * kOp);
    tma_load_tile<HD>(sKV, &p.tmap_qkv, &bar_kv[0], colK, kb_first * kBlk);
    tma_load_tile<HD>(sKV + kOp, &p.tmap_qkv, &bar_kv[0], colV, kb_first * kBlk);
  }

  constexpr uint32_t idesc_s = make_idesc(kFmtBF16, kFmtBF16, false, false, 128, 128);
  constexpr uint32_t idesc_o = make_idesc(kFmtBF16, kFmtBF16, false, true, 128, HD);
  const float sl2 = p.scale * kLog2e;
  const uint32_t dthr = p.drop.thr, rowkey = attn_row_key(p, h, row_tok);
  float m_run = -CUDART_INF_F, l_run = 0.f;
  float acc[HD];
#pragma unroll
  for (int i = 0; i < HD; ++i) acc[i] = 0.f;

  mbar_wait(bar_q, 0);
  for (int it = 0; it < nkb; ++it) {
    const int st = it & 1;
    const int k0 = (kb_first + it) * kBlk;
    uint8_t* sK = sKV + st * 2 * kOp;
    uint8_t* sV = sK + kOp;
    if (tid == 0) {
      if (it + 1 < nkb) {  // prefetch the next K/V block into the other stage (its readers finished last iteration)
        uint8_t* nK = sKV + (st ^ 1) * 2 * kOp;
        mbar_expect_tx(&bar_kv[st ^ 1], 2 * kOp);
        tma_load_tile<HD>(nK, &p.tmap_qkv, &bar_kv[st ^ 1], colK, k0 + kBlk);
        tma_load_tile<HD>(nK + kOp, &p.tmap_qkv, &bar_kv[st ^ 1], colV, k0 + kBlk);
      }
      mbar_wait(&bar_kv[st], (it >> 1) & 1);
      tc_fence_after();
      const uint64_t dq = make_smem_desc(smem_u32(sQ), 16, 1024);
      const uint64_t dk = make_smem_desc(smem_u32(sK), 16, 1024);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tS, dq + kstep_off(k), dk + kstep_off(k), idesc_s, k > 0);
      umma_commit(bar_s);
    }
    mbar_wait(bar_s, it & 1);
    tc_fence_after();
    // ---- softmax over this thread's row: pass 1 = masked row max, pass 2 = exp / sum / write P ----
    const int c_lo = seq_start - k0, c_hi = row_last_key(p, row_tok) - k0;  // valid columns: c_lo <= c <= c_hi
    float mx = -CUDART_INF_F;
#pragma unroll 1
    for (int ch = 0; ch < 4; ++ch) {
      const uint32_t vm = chunk_mask(c_lo, c_hi, ch);
      if (!__any_sync(kFullWarp, vm != 0u)) continue;  // warp-uniform: tcgen05.ld is a warp-collective
      float s[32];
      tmem_ld32(tS + lane_off + ch * 32, s);
      mx = fmaxf(mx, __all_sync(kFullWarp, vm == kFullWarp) ? chunk_rowmax<false>(s, vm) : chunk_rowmax<true>(s, vm));
    }
    const float m_new = fmaxf(m_run, mx * sl2);
    const float m_ref = (m_new == -CUDART_INF_F) ? 0.f : m_new;
    const float alpha = ex2_fast(m_run - m_ref);  // m_run = -inf -> 0
    float lsum = 0.f;
#pragma unroll 1
    for (int ch = 0; ch < 4; ++ch) {
      const uint32_t vm = chunk_mask(c_lo, c_hi, ch);
      uint8_t* atom = sP + (ch >> 1) * kTile;
      if (!__any_sync(kFullWarp, vm != 0u)) {  // beyond the diagonal for every row of this warp: P = 0
#pragma unroll
        for (int v = 0; v < 4; ++v) st_swz(atom, tid, (ch & 1) * 4 + v, make_uint4(0, 0, 0, 0));
        continue;
      }
      float s[32];
      tmem_ld32(tS + lane_off + ch * 32, s);
      lsum += __all_sync(kFullWarp, vm == kFullWarp) ? chunk_exp<false>(s, vm, sl2, m_ref) : chunk_exp<true>(s, vm, sl2, m_ref);
      if (dthr) drop_p32(s, rowkey, k0 + ch * 32, dthr, p.drop.scale);
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        uint4 q;
        q.x = pack2(s[v * 8 + 0], s[v * 8 + 1]); q.y = pack2(s[v * 8 + 2], s[v * 8 + 3]);
        q.z = pack2(s[v * 8 + 4], s[v * 8 + 5]); q.w = pack2(s[v * 8 + 6], s[v * 8 + 7]);
        st_swz(atom, tid, (ch & 1) * 4 + v, q);
      }
    }
    l_run = l_run * alpha + lsum;
    m_run = m_new;
#pragma unroll
    for (int i = 0; i < HD; ++i) acc[i] *= alpha;
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < kBlk / 16; ++k) {
        const uint64_t dp = make_smem_desc(smem_u32(sP) + (k >> 2) * kTile + (k & 3) * 32, 16, 1024);
        const uint64_t dv = make_smem_desc(smem_u32(sV) + k * 2048, kTile, 1024);
        umma_f16(tO, dp, dv, idesc_o, k > 0);
      }
      umma_commit(bar_o);
    }
    mbar_wait(bar_o, it & 1);
    tc_fence_after();
#pragma unroll
    for (int ch = 0; ch < HD / 32; ++ch) {
      float o[32];
      tmem_ld32(tO + lane_off + ch * 32, o);
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[ch * 32 + i] += o[i];
    }
    tc_fence_before();  // order this iteration's TMEM reads before the next iteration's MMA writes
    __syncthreads();
  }
  // ---- epilogue: O tile staged (swizzled) in the Q tile -- every MMA that read it has completed -- and stored by TMA ----
  {
    const float inv = l_run > 0.f ? 1.f / l_run : 0.f;  // rows >= M: all masked -> zeros, clipped by the tensor map anyway
#pragma unroll
    for (int v = 0; v < HD / 8; ++v) {
      uint4 q;
      q.x = pack2(acc[v * 8 + 0] * inv, acc[v * 8 + 1] * inv); q.y = pack2(acc[v * 8 + 2] * inv, acc[v * 8 + 3] * inv);
      q.z = pack2(acc[v * 8 + 4] * inv, acc[v * 8 + 5] * inv); q.w = pack2(acc[v * 8 + 6] * inv, acc[v * 8 + 7] * inv);
      st_swz(sQ + (v >> 3) * kTile, tid, v & 7, q);
    }
    fence_proxy_async_smem();
    if (row_tok < p.M && p.lse) {
      const int b = row_tok / p.T, t = row_tok % p.T;
      p.lse[(size_t(b) * p.H + h) * p.T + t] = (m_run + log2f(l_run)) * 0.6931471805599453f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    if (elect_one()) {
      tma_store_tile<HD>(&p.tmap_out, sQ, h * HD, q0);
      tma_store_commit();
      tma_store_wait_read<0>();
    }
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------------
// Common inner step for a (q-block i, kv-block j, head h) pair, executed by 128 threads (thread = q row):
//   S = Q K^T, dP = dO V^T  (tensor cores)  ->  P = exp2(S*sl2 - lse*log2e),  dS = P * (dP - D) * scale
//   P and dS are written as bf16 into swizzled smem tiles.
template <bool WRITE_P>
DTB_DEVICE void bwd_softmax_tiles(uint32_t tS, uint32_t tDP, uint32_t lane_off, int tid, int c_lo, int c_hi, float sl2,
                                  float lse_l2, float Drow, float scale, uint8_t* sP, uint8_t* sDS, uint32_t rowkey, int k0,
                                  uint32_t dthr, float dscale, int ch_lo = 0, int ch_hi = 3) {
  const float nD = -Drow * scale;
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    const uint32_t vm = chunk_mask(c_lo, c_hi, ch);
    // warp-uniformly masked chunk (see attn_fwd_small_kernel; the vote also covers the tiled kernels' diagonal blocks): P = dS = 0
    if (ch < ch_lo || ch > ch_hi || !__any_sync(kFullWarp, vm != 0u)) {
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        if (WRITE_P) st_swz(sP + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, make_uint4(0, 0, 0, 0));
        st_swz(sDS + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, make_uint4(0, 0, 0, 0));
      }
      continue;
    }
    float s[32], dp[32];
    tmem_ld32x2(tS + lane_off + ch * 32, s, tDP + lane_off + ch * 32, dp);  // both loads in flight, one wait
    const bool all = __all_sync(kFullWarp, vm == kFullWarp);
    if (dthr) {  // dropout on P: dV uses the masked P, dS = P * (mask * dP - D) * scale  (D = rowsum(dO * O) is unchanged)
      float mk[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) mk[i] = 1.f;
      drop_p32(mk, rowkey, k0 + ch * 32, dthr, dscale);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float e = ex2_fast(fmaf(s[i], sl2, -lse_l2));
        const float pv = (all || ((vm >> i) & 1u)) ? e : 0.f;
        s[i] = pv * mk[i];
        dp[i] = pv * fmaf(dp[i] * mk[i], scale, nD);
      }
    } else if (all) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float pv = ex2_fast(fmaf(s[i], sl2, -lse_l2));
        s[i] = pv;
        dp[i] = pv * fmaf(dp[i], scale, nD);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float pv = ((vm >> i) & 1u) ? ex2_fast(fmaf(s[i], sl2, -lse_l2)) : 0.f;
        s[i] = pv;
        dp[i] = pv * fmaf(dp[i], scale, nD);
      }
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      uint4 q;
      if (WRITE_P) {
        q.x = pack2(s[v * 8 + 0], s[v * 8 + 1]); q.y = pack2(s[v * 8 + 2], s[v * 8 + 3]);
        q.z = pack2(s[v * 8 + 4], s[v * 8 + 5]); q.w = pack2(s[v * 8 + 6], s[v * 8 + 7]);
        st_swz(sP + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, q);
      }
      q.x = pack2(dp[v * 8 + 0], dp[v * 8 + 1]); q.y = pack2(dp[v * 8 + 2], dp[v * 8 + 3]);
      q.z = pack2(dp[v * 8 + 4], dp[v * 8 + 5]); q.w = pack2(dp[v * 8 + 6], dp[v * 8 + 7]);
      st_swz(sDS + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, q);
    }
  }
}

// D = rowsum(dO * O), lse in log2 units, for this thread's q row
template <int HD>
DTB_DEVICE void load_row_stats(const AttnParams& p, int row_tok, int h, float& Drow, float& lse_l2) {
  Drow = 0.f;
  lse_l2 = 0.f;
  if (row_tok < p.M) {
    const uint4* a = reinterpret_cast<const uint4*>(p.dout + size_t(row_tok) * p.ld_o + h * HD);
    const uint4* b = reinterpret_cast<const uint4*>(p.o + size_t(row_tok) * p.ld_o + h * HD);
#pragma unroll
    for (int v = 0; v < HD / 8; ++v) {
      const uint4 x = __ldg(a + v), y = __ldg(b + v);
      const __nv_bfloat162* xh = reinterpret_cast<const __nv_bfloat162*>(&x);
      const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&y);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 fx = __bfloat1622float2(xh[k]), fy = __bfloat1622float2(yh[k]);
        Drow += fx.x * fy.x + fx.y * fy.y;
      }
    }
    const int b_ = row_tok / p.T, t = row_tok % p.T;
    lse_l2 = p.lse[(size_t(b_) * p.H + h) * p.T + t] * kLog2e;
  }
}

// Same statistics from the TMA-loaded dO / O tiles in shared memory (128B-swizzled [128 x HD] bf16): replaces 16 row-strided
// LDG.128 per thread (17 % of the single-block kernel's stall samples sat on their first use) with conflict-free LDS.
template <int HD>
DTB_DEVICE void row_stats_smem(const AttnParams& p, const uint8_t* sDO, const uint8_t* sO, int row, int row_tok, int h, float& Drow,
                               float& lse_l2) {
  Drow = 0.f;
  lse_l2 = 0.f;
#pragma unroll
  for (int ch = 0; ch < HD / 8; ++ch) {
    const uint32_t off = (ch >> 3) * kTile + row * 128 + (((ch & 7) ^ (row & 7)) << 4);
    const uint4 x = *reinterpret_cast<const uint4*>(sDO + off), y = *reinterpret_cast<const uint4*>(sO + off);
    const __nv_bfloat162* xh = reinterpret_cast<const __nv_bfloat162*>(&x);
    const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&y);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 fx = __bfloat1622float2(xh[k]), fy = __bfloat1622float2(yh[k]);
      Drow += fx.x * fy.x + fx.y * fy.y;
    }
  }
  if (row_tok < p.M) {
    const int b_ = row_tok / p.T, t = row_tok % p.T;
    lse_l2 = p.lse[(size_t(b_) * p.H + h) * p.T + t] * kLog2e;
  }
}

// --- KV-owner kernel: grid (kv-block, kv-head).  smem: K V | (Q dO) x stages | P(2) | dS(2)
//     hd 64: 32 + 2 x 32 + 32 + 32 = 160 KB;  hd 128: 64 + 1 x 64 + 32 + 32 = 192 KB (two Q/dO stages would need 256 KB)
// TMEM: S[128] dP[128] dV[hd] dK[hd] -> 512 columns at hd 128 (all of them)
template <int HD>
constexpr int bwd_kv_stages() { return HD == 64 ? 2 : 1; }
template <int HD>
constexpr int bwd_kv_smem() { return 1024 + kTile * (2 * (HD / 64) + bwd_kv_stages<HD>() * 2 * (HD / 64) + 4) + 128; }
static_assert(bwd_kv_smem<64>() <= kSmemLimit && bwd_kv_smem<128>() <= kSmemLimit, "attn_bwd_kv smem budget");
static_assert(256 + 2 * 128 <= 512, "attn_bwd_kv TMEM budget");

template <int HD>
__global__ void __launch_bounds__(128, 1) attn_bwd_kv_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kOp = kTile * (HD / 64), kSt = bwd_kv_stages<HD>();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // PDL: a dependent GEMM may start its prologue (sm100_ptx.cuh)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = smem + kOp;
  uint8_t* sQD = smem + 2 * kOp;  // [kSt stages][Q, dO]
  uint8_t* sP = sQD + kSt * 2 * kOp;
  uint8_t* sDS = sP + 2 * kTile;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * kTile);
  uint64_t* bar_kv = bars;
  uint64_t* bar_qd = bars + 1;  // [2] (one used with a single stage)
  uint64_t* bar_s = bars + 3;
  uint64_t* bar_g = bars + 4;   // dV/dK MMAs of this iteration done (P/dS/Q/dO buffers reusable)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x, warp = tid >> 5;
  int kb, hk;
  lpt_block(p, false, kb, hk);
  const int group = p.H / p.Hkv;
  const int k0 = kb * kBlk;
  // q blocks that can attend into this kv block: from kb up to the block holding the end of the last key's sequence
  const int last_key = min(k0 + kBlk, p.M) - 1;
  const int seq_end = (last_key / p.T + 1) * p.T;  // exclusive
  const int qb_last = (min(seq_end, p.M) - 1) / kBlk;
  const int nqb = qb_last - kb + 1;
  const int niter = nqb * group;
  const int colK = (p.H + hk) * HD, colV = (p.H + p.Hkv + hk) * HD;

  if (tid == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    tma_prefetch_desc(&p.tmap_do);
    mbar_init(bar_kv, 1);
    mbar_init(&bar_qd[0], 1);
    mbar_init(&bar_qd[1], 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_g, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  const uint32_t tS = tmem, tDP = tmem + 128, tDV = tmem + 256, tDK = tmem + 256 + HD;
  const uint32_t lane_off = (uint32_t(warp) * 32u) << 16;

  auto issue_qd = [&](int it) {
    const int st = kSt == 2 ? (it & 1) : 0;
    const int hq = hk * group + it % group;
    const int q0 = (kb + it / group) * kBlk;
    uint8_t* dst = sQD + st * 2 * kOp;
    mbar_expect_tx(&bar_qd[st], 2 * kOp);
    tma_load_tile<HD>(dst, &p.tmap_qkv, &bar_qd[st], hq * HD, q0);
    tma_load_tile<HD>(dst + kOp, &p.tmap_do, &bar_qd[st], hq * HD, q0);
  };
  if (tid == 0) {
    mbar_expect_tx(bar_kv, 2 * kOp);
    tma_load_tile<HD>(sK, &p.tmap_qkv, bar_kv, colK, k0);
    tma_load_tile<HD>(sV, &p.tmap_qkv, bar_kv, colV, k0);
    issue_qd(0);
  }
  constexpr uint32_t idesc_s = make_idesc(kFmtBF16, kFmtBF16, false, false, 128, 128);   // S, dP
  constexpr uint32_t idesc_g = make_idesc(kFmtBF16, kFmtBF16, true, true, 128, HD);      // dV = P^T dO, dK = dS^T Q
  const float sl2 = p.scale * kLog2e;
  mbar_wait(bar_kv, 0);

  for (int it = 0; it < niter; ++it) {
    const int st = kSt == 2 ? (it & 1) : 0;
    const int hq = hk * group + it % group;
    const int q0 = (kb + it / group) * kBlk;
    uint8_t* sQ = sQD + st * 2 * kOp;
    uint8_t* sDO = sQ + kOp;
    if (tid == 0) {
      if (kSt == 2 && it + 1 < niter) issue_qd(it + 1);  // other stage: its MMAs completed (bar_g of iteration it-1)
      mbar_wait(&bar_qd[st], kSt == 2 ? ((it >> 1) & 1) : (it & 1));
      tc_fence_after();
      const uint64_t dq = make_smem_desc(smem_u32(sQ), 16, 1024), dk = make_smem_desc(smem_u32(sK), 16, 1024);
      const uint64_t ddo = make_smem_desc(smem_u32(sDO), 16, 1024), dv = make_smem_desc(smem_u32(sV), 16, 1024);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tS, dq + kstep_off(k), dk + kstep_off(k), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tDP, ddo + kstep_off(k), dv + kstep_off(k), idesc_s, k > 0);
      umma_commit(bar_s);
    }
    const int row_tok = q0 + tid;
    float Drow, lse_l2;
    load_row_stats<HD>(p, row_tok, hq, Drow, lse_l2);
    const int seq_start = (row_tok / p.T) * p.T;
    const int c_lo = seq_start - k0, c_hi = row_last_key(p, row_tok) - k0;
    mbar_wait(bar_s, it & 1);
    tc_fence_after();
    bwd_softmax_tiles<true>(tS, tDP, lane_off, tid, c_lo, c_hi, sl2, lse_l2, Drow, p.scale, sP, sDS, attn_row_key(p, hq, row_tok), k0,
                            p.drop.thr, p.drop.scale);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      // A = P^T / dS^T: MN-major (m = key, 2 atoms of 64 keys, LBO = atom stride), k = q rows (16 rows = 2048 B per step)
      // B = dO / Q   : MN-major (n = hd, one atom), k = q rows
#pragma unroll
      for (int k = 0; k < kBlk / 16; ++k) {
        const uint64_t a1 = make_smem_desc(smem_u32(sP) + k * 2048, kTile, 1024);
        const uint64_t b1 = make_smem_desc(smem_u32(sDO) + k * 2048, kTile, 1024);
        umma_f16(tDV, a1, b1, idesc_g, (it > 0 || k > 0));
      }
#pragma unroll
      for (int k = 0; k < kBlk / 16; ++k) {
        const uint64_t a2 = make_smem_desc(smem_u32(sDS) + k * 2048, kTile, 1024);
        const uint64_t b2 = make_smem_desc(smem_u32(sQ) + k * 2048, kTile, 1024);
        umma_f16(tDK, a2, b2, idesc_g, (it > 0 || k > 0));
      }
      umma_commit(bar_g);
    }
    mbar_wait(bar_g, it & 1);  // smem tiles + S/dP TMEM free for the next iteration
    tc_fence_after();
    if (kSt == 1 && tid == 0 && it + 1 < niter) issue_qd(it + 1);  // single stage: refill once this iteration's MMAs are done
  }
  // ---- write dK, dV (thread = key row).  tcgen05.ld is warp-collective: loads are unconditional, stores guarded ----
  const int key_tok = k0 + tid;
#pragma unroll 1
  for (int which = 0; which < 2; ++which) {
    const uint32_t t = which == 0 ? tDK : tDV;
    __nv_bfloat16* dst = p.out + size_t(key_tok) * p.ld_out + (which == 0 ? colK : colV);
#pragma unroll
    for (int ch = 0; ch < HD / 32; ++ch) {
      float o[32];
      tmem_ld32(t + lane_off + ch * 32, o);
      if (key_tok < p.M) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          uint4 q;
          q.x = pack2(o[v * 8 + 0], o[v * 8 + 1]); q.y = pack2(o[v * 8 + 2], o[v * 8 + 3]);
          q.z = pack2(o[v * 8 + 4], o[v * 8 + 5]); q.w = pack2(o[v * 8 + 6], o[v * 8 + 7]);
          reinterpret_cast<uint4*>(dst)[ch * 4 + v] = q;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// --- Q-owner kernel: grid (q-block, head).  smem: Q dO | (K V) x2 | dS(2) = 32+64+32 = 128 KB (hd 128: 64+128+32 = 224 KB) ---
// TMEM: S[128] dP[128] dQ[hd] -> 512 columns allocated
template <int HD>
constexpr int bwd_q_smem() { return 1024 + kTile * (6 * (HD / 64) + 2) + 128; }
static_assert(bwd_q_smem<64>() <= kSmemLimit && bwd_q_smem<128>() <= kSmemLimit, "attn_bwd_q smem budget");

template <int HD>
__global__ void __launch_bounds__(128, 1) attn_bwd_q_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kOp = kTile * (HD / 64);
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // PDL: a dependent GEMM may start its prologue (sm100_ptx.cuh)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sDO = smem + kOp;
  uint8_t* sKV = smem + 2 * kOp;
  uint8_t* sDS = smem + 6 * kOp;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * kTile);
  uint64_t* bar_q = bars;
  uint64_t* bar_kv = bars + 1;  // [2]
  uint64_t* bar_s = bars + 3;
  uint64_t* bar_g = bars + 4;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x, warp = tid >> 5;
  int qb, h;
  lpt_block(p, true, qb, h);
  const int hk = h / (p.H / p.Hkv);
  const int q0 = qb * kBlk;
  const int row_tok = q0 + tid;
  const int seq_start = (row_tok / p.T) * p.T;
  const int kb_first = ((q0 / p.T) * p.T) / kBlk;
  const int nkb = qb - kb_first + 1;
  const int colK = (p.H + hk) * HD, colV = (p.H + p.Hkv + hk) * HD;

  if (tid == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    tma_prefetch_desc(&p.tmap_do);
    mbar_init(bar_q, 1);
    mbar_init(&bar_kv[0], 1);
    mbar_init(&bar_kv[1], 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_g, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  const uint32_t tS = tmem, tDP = tmem + 128, tDQ = tmem + 256;
  const uint32_t lane_off = (uint32_t(warp) * 32u) << 16;

  if (tid == 0) {
    mbar_expect_tx(bar_q, 2 * kOp);
    tma_load_tile<HD>(sQ, &p.tmap_qkv, bar_q, h * HD, q0);
    tma_load_tile<HD>(sDO, &p.tmap_do, bar_q, h * HD, q0);
    mbar_expect_tx(&bar_kv[0], 2 * kOp);
    tma_load_tile<HD>(sKV, &p.tmap_qkv, &bar_kv[0], colK, kb_first * kBlk);
    tma_load_tile<HD>(sKV + kOp, &p.tmap_qkv, &bar_kv[0], colV, kb_first * kBlk);
  }
  constexpr uint32_t idesc_s = make_idesc(kFmtBF16, kFmtBF16, false, false, 128, 128);
  constexpr uint32_t idesc_q = make_idesc(kFmtBF16, kFmtBF16, false, true, 128, HD);  // dQ = dS K  (B = K, MN-major)
  const float sl2 = p.scale * kLog2e;
  const uint32_t rowkey = attn_row_key(p, h, row_tok);
  float Drow, lse_l2;
  load_row_stats<HD>(p, row_tok, h, Drow, lse_l2);
  mbar_wait(bar_q, 0);

  for (int it = 0; it < nkb; ++it) {
    const int st = it & 1;
    const int k0 = (kb_first + it) * kBlk;
    uint8_t* sK = sKV + st * 2 * kOp;
    uint8_t* sV = sK + kOp;
    if (tid == 0) {
      if (it + 1 < nkb) {
        uint8_t* nK = sKV + (st ^ 1) * 2 * kOp;
        mbar_expect_tx(&bar_kv[st ^ 1], 2 * kOp);
        tma_load_tile<HD>(nK, &p.tmap_qkv, &bar_kv[st ^ 1], colK, k0 + kBlk);
        tma_load_tile<HD>(nK + kOp, &p.tmap_qkv, &bar_kv[st ^ 1], colV, k0 + kBlk);
      }
      mbar_wait(&bar_kv[st], (it >> 1) & 1);
      tc_fence_after();
      const uint64_t dq = make_smem_desc(smem_u32(sQ), 16, 1024), dk = make_smem_desc(smem_u32(sK), 16, 1024);
      const uint64_t ddo = make_smem_desc(smem_u32(sDO), 16, 1024), dv = make_smem_desc(smem_u32(sV), 16, 1024);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tS, dq + kstep_off(k), dk + kstep_off(k), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tDP, ddo + kstep_off(k), dv + kstep_off(k), idesc_s, k > 0);
      umma_commit(bar_s);
    }
    const int c_lo = seq_start - k0, c_hi = row_last_key(p, row_tok) - k0;
    mbar_wait(bar_s, it & 1);
    tc_fence_after();
    bwd_softmax_tiles<false>(tS, tDP, lane_off, tid, c_lo, c_hi, sl2, lse_l2, Drow, p.scale, nullptr, sDS, rowkey, k0, p.drop.thr,
                             p.drop.scale);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < kBlk / 16; ++k) {
        const uint64_t a = make_smem_desc(smem_u32(sDS) + (k >> 2) * kTile + (k & 3) * 32, 16, 1024);  // dS K-major
        const uint64_t b = make_smem_desc(smem_u32(sK) + k * 2048, kTile, 1024);                       // K MN-major
        umma_f16(tDQ, a, b, idesc_q, (it > 0 || k > 0));
      }
      umma_commit(bar_g);
    }
    mbar_wait(bar_g, it & 1);
    tc_fence_after();
  }
#pragma unroll
  for (int c2 = 0; c2 < HD / 64; ++c2) {
    float o0[32], o1[32];
    tmem_ld32(tDQ + lane_off + c2 * 64, o0);
    tmem_ld32(tDQ + lane_off + c2 * 64 + 32, o1);
    if (row_tok < p.M) {
      __nv_bfloat16* dst = p.out + size_t(row_tok) * p.ld_out + h * HD + c2 * 64;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        uint4 q;
        q.x = pack2(o0[v * 8 + 0], o0[v * 8 + 1]); q.y = pack2(o0[v * 8 + 2], o0[v * 8 + 3]);
        q.z = pack2(o0[v * 8 + 4], o0[v * 8 + 5]); q.w = pack2(o0[v * 8 + 6], o0[v * 8 + 7]);
        reinterpret_cast<uint4*>(dst)[v] = q;
        q.x = pack2(o1[v * 8 + 0], o1[v * 8 + 1]); q.y = pack2(o1[v * 8 + 2], o1[v * 8 + 3]);
        q.z = pack2(o1[v * 8 + 4], o1[v * 8 + 5]); q.w = pack2(o1[v * 8 + 6], o1[v * 8 + 7]);
        reinterpret_cast<uint4*>(dst)[4 + v] = q;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// single-block fast paths: every 128-token block is self-contained (128 % T == 0 or T == 128: the reference miner's T = 64)
// ------------------------------------------------------------------------------------------------------------------
// forward: Q K V | P aliases the first two atoms (Q+K at hd 64, Q at hd 128: dead once S is computed);  TMEM: S[128], O reuses
// S[0:hd]  -> hd 64: 48 KB + 128 columns, four CTAs per SM overlap each other's TMA / MMA / softmax phases; hd 128: 96 KB, two.
template <int HD>
constexpr int fwd_small_smem() { return 1024 + kTile * 3 * (HD / 64) + 64; }
static_assert(fwd_small_smem<64>() <= kSmemLimit / 4 && fwd_small_smem<128>() <= kSmemLimit / 2, "attn_fwd_small smem budget");

template <int HD>
__global__ void __launch_bounds__(128, HD == 64 ? 4 : 2) attn_fwd_small_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kOp = kTile * (HD / 64);
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // PDL: a dependent GEMM may start its prologue (sm100_ptx.cuh)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + kOp;
  uint8_t* sV = smem + 2 * kOp;
  uint8_t* sP = smem;  // 2 atoms over Q|K (hd 64) or Q (hd 128)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOp * 3);
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 3);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int qb = blockIdx.x, h = blockIdx.y;
  const int hk = h / (p.H / p.Hkv);
  const int q0 = qb * kBlk;
  const int row_tok = q0 + tid;
  if (tid == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();  // PDL: launched early -- everything above touched only shared memory / TMEM / kernel parameters
  const uint32_t tmem = *tmem_ptr;
  const uint32_t lane_off = (uint32_t(warp) * 32u) << 16;
  constexpr uint32_t idesc_s = make_idesc(kFmtBF16, kFmtBF16, false, false, 128, 128);
  constexpr uint32_t idesc_o = make_idesc(kFmtBF16, kFmtBF16, false, true, 128, HD);
  if (warp == 0) {  // warp-uniform issue: only the instructions themselves sit under elect.sync (see sm100_gemm.cu)
    if (elect_one()) {
      mbar_expect_tx(&bars[0], 3 * kOp);
      tma_load_tile<HD>(sQ, &p.tmap_qkv, &bars[0], h * HD, q0);
      tma_load_tile<HD>(sK, &p.tmap_qkv, &bars[0], (p.H + hk) * HD, q0);
      tma_load_tile<HD>(sV, &p.tmap_qkv, &bars[0], (p.H + p.Hkv + hk) * HD, q0);
    }
    mbar_wait(&bars[0], 0);
    tc_fence_after();
    const uint64_t dq = make_smem_desc(smem_u32(sQ), 16, 1024), dk = make_smem_desc(smem_u32(sK), 16, 1024);
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tmem, dq + kstep_off(k), dk + kstep_off(k), idesc_s, k > 0);
      umma_commit(&bars[1]);
    }
  }
  const int c_lo = (row_tok / p.T) * p.T - q0, c_hi = row_last_key(p, row_tok) - q0;
  // 32-column chunks this WARP has to look at: with T % 32 == 0 all 32 rows of a warp sit in one sequence, so the chunks left
  // of the sequence start and right of the warp's last row are masked for every lane (T = 64: 1.5 of 4 chunks on average).
  int ch_lo = 0, ch_hi = 3;
  if (p.T % 32 == 0) {
    ch_lo = c_lo >> 5;  // c_lo is warp-uniform and a multiple of 32
    ch_hi = warp;       // columns beyond the warp's last row (warp * 32 + 31) are causal-masked
  }
  const float sl2 = p.scale * kLog2e;
  const uint32_t rowkey = attn_row_key(p, h, row_tok);
  mbar_wait(&bars[1], 0);
  tc_fence_after();
  float mx = -CUDART_INF_F;
#pragma unroll 1
  for (int ch = ch_lo; ch <= ch_hi; ++ch) {
    const uint32_t vm = chunk_mask(c_lo, c_hi, ch);
    if (!__any_sync(kFullWarp, vm != 0u)) continue;
    float sv[32];
    tmem_ld32(tmem + lane_off + ch * 32, sv);
    mx = fmaxf(mx, __all_sync(kFullWarp, vm == kFullWarp) ? chunk_rowmax<false>(sv, vm) : chunk_rowmax<true>(sv, vm));
  }
  const float m_ref = mx == -CUDART_INF_F ? 0.f : mx * sl2;  // fully masked row (rows >= M): P = 0, no NaN
  float lsum = 0.f;
#pragma unroll 1
  for (int ch = 0; ch < 4; ++ch) {
    const uint32_t vm = chunk_mask(c_lo, c_hi, ch);
    if (ch < ch_lo || ch > ch_hi || !__any_sync(kFullWarp, vm != 0u)) {  // fully masked for this warp: P = 0
#pragma unroll
      for (int v = 0; v < 4; ++v) st_swz(sP + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, make_uint4(0, 0, 0, 0));
      continue;
    }
    float sv[32];
    tmem_ld32(tmem + lane_off + ch * 32, sv);
    lsum += __all_sync(kFullWarp, vm == kFullWarp) ? chunk_exp<false>(sv, vm, sl2, m_ref) : chunk_exp<true>(sv, vm, sl2, m_ref);
    if (p.drop.thr) drop_p32(sv, rowkey, q0 + ch * 32, p.drop.thr, p.drop.scale);
    // all 128 threads finished READING Q/K? they are only read by the tensor core, which completed (bars[1]) -> safe
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      uint4 q;
      q.x = pack2(sv[v * 8 + 0], sv[v * 8 + 1]); q.y = pack2(sv[v * 8 + 2], sv[v * 8 + 3]);
      q.z = pack2(sv[v * 8 + 4], sv[v * 8 + 5]); q.w = pack2(sv[v * 8 + 6], sv[v * 8 + 7]);
      st_swz(sP + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, q);
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    const uint32_t pbase = smem_u32(sP), vbase = smem_u32(sV);
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < kBlk / 16; ++k) {
        const uint64_t dp = make_smem_desc(pbase + (k >> 2) * kTile + (k & 3) * 32, 16, 1024);
        const uint64_t dv = make_smem_desc(vbase + k * 2048, kTile, 1024);
        umma_f16(tmem, dp, dv, idesc_o, k > 0);  // O overwrites S[0:hd] (every thread has consumed S)
      }
      umma_commit(&bars[2]);
    }
  }
  mbar_wait(&bars[2], 0);
  tc_fence_after();
  const float inv = lsum > 0.f ? 1.f / lsum : 0.f;
  // O tile -> swizzled staging tile in the (dead) Q region -> ONE TMA store (rows >= M are clipped by the tensor map).
  // Per-thread 16 B global stores of 32 different rows per instruction throttled the LSU (lg_throttle, ncu).
#pragma unroll
  for (int ch = 0; ch < HD / 32; ++ch) {
    float o[32];
    tmem_ld32(tmem + lane_off + ch * 32, o);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      uint4 q;
      q.x = pack2(o[v * 8 + 0] * inv, o[v * 8 + 1] * inv); q.y = pack2(o[v * 8 + 2] * inv, o[v * 8 + 3] * inv);
      q.z = pack2(o[v * 8 + 4] * inv, o[v * 8 + 5] * inv); q.w = pack2(o[v * 8 + 6] * inv, o[v * 8 + 7] * inv);
      st_swz(sQ + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, q);
    }
  }
  fence_proxy_async_smem();
  if (row_tok < p.M && p.lse) {
    const int b = row_tok / p.T, t = row_tok % p.T;
    p.lse[(size_t(b) * p.H + h) * p.T + t] = (m_ref + log2f(lsum)) * 0.6931471805599453f;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    if (elect_one()) {
      tma_store_tile<HD>(&p.tmap_out, sQ, h * HD, q0);
      tma_store_commit();
      tma_store_wait_read<0>();  // the staging tile must outlive the bulk read
    }
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem, 128);
  }
}

// backward, all five products in ONE CTA (no recomputation across kernels):
//   S = Q K^T, dP = dO V^T  ->  P, dS  ->  dV = P^T dO, dK = dS^T Q, dQ = dS K.     (MHA only: H == Hkv)
// smem: Q K dO | V -> P0 | P1 | dS(2) = 112 KB (P overwrites V, which is dead once dP is computed);
// TMEM: S[128] dP[128], then dV/dK/dQ overwrite them (every thread has consumed S/dP) = 256 columns -> TWO CTAs per SM
// overlap each other's TMA / MMA / softmax phases (the first version ran one CTA per SM at 6 % occupancy, 126 us/layer).
// hd 128: Q K dO | V = P(2) | dS(2) = 160 KB; dV/dK/dQ take 384 columns -> 512 allocated, one CTA per SM.
template <int HD>
constexpr int bwd_small_smem() { return kTile * (3 * (HD / 64) + 4) + 64; }
static_assert(bwd_small_smem<64>() <= kSmemLimit / 2 && bwd_small_smem<128>() <= kSmemLimit, "attn_bwd_small smem budget");

template <int HD>
__global__ void __launch_bounds__(128, HD == 64 ? 2 : 1) attn_bwd_small_kernel(const __grid_constant__ AttnParams p) {
  constexpr int kOp = kTile * (HD / 64);
  constexpr uint32_t kCols = HD == 64 ? 256 : 512;  // TMEM columns
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // PDL: a dependent GEMM may start its prologue (sm100_ptx.cuh)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;  // the dynamic window starts 1 KB-aligned (no static shared memory in this kernel)
  uint8_t* sQ = smem;
  uint8_t* sK = smem + kOp;
  uint8_t* sDO = smem + 2 * kOp;
  uint8_t* sV = smem + 3 * kOp;
  uint8_t* sP = smem + 3 * kOp;     // aliases V
  uint8_t* sDS = sP + 2 * kTile;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * kTile);
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 3);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int qb = blockIdx.x, h = blockIdx.y;
  const int q0 = qb * kBlk;
  const int row_tok = q0 + tid;
  const int colQ = h * HD, colK = (p.H + h) * HD, colV = (2 * p.H + h) * HD;
  if (tid == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    tma_prefetch_desc(&p.tmap_do);
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, kCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();  // PDL: launched early -- everything above touched only shared memory / TMEM / kernel parameters
  const uint32_t tmem = *tmem_ptr;
  const uint32_t tS = tmem, tDP = tmem + 128;
  const uint32_t tDV = tmem, tDK = tmem + HD, tDQ = tmem + 2 * HD;  // reuse S / dP after the softmax tiles are in smem
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();  // layout assumption of the swizzled tiles
  const uint32_t lane_off = (uint32_t(warp) * 32u) << 16;
  constexpr uint32_t idesc_s = make_idesc(kFmtBF16, kFmtBF16, false, false, 128, 128);
  constexpr uint32_t idesc_g = make_idesc(kFmtBF16, kFmtBF16, true, true, 128, HD);
  constexpr uint32_t idesc_q = make_idesc(kFmtBF16, kFmtBF16, false, true, 128, HD);
  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(&bars[0], 5 * kOp);
      tma_load_tile<HD>(sQ, &p.tmap_qkv, &bars[0], colQ, q0);
      tma_load_tile<HD>(sK, &p.tmap_qkv, &bars[0], colK, q0);
      tma_load_tile<HD>(sV, &p.tmap_qkv, &bars[0], colV, q0);
      tma_load_tile<HD>(sDO, &p.tmap_do, &bars[0], colQ, q0);
      tma_load_tile<HD>(sDS, &p.tmap_o, &bars[0], colQ, q0);  // O tile parks in the (still dead) dS region until D is formed
    }
    mbar_wait(&bars[0], 0);
    tc_fence_after();
    const uint64_t dq = make_smem_desc(smem_u32(sQ), 16, 1024), dk = make_smem_desc(smem_u32(sK), 16, 1024);
    const uint64_t ddo = make_smem_desc(smem_u32(sDO), 16, 1024), dv = make_smem_desc(smem_u32(sV), 16, 1024);
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tS, dq + kstep_off(k), dk + kstep_off(k), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_f16(tDP, ddo + kstep_off(k), dv + kstep_off(k), idesc_s, k > 0);
      umma_commit(&bars[1]);
    }
  }
  float Drow, lse_l2;
  if (warp != 0) mbar_wait(&bars[0], 0);  // (warp 0 passed it before issuing the MMAs) the dO / O tiles have landed
  // each thread reads ITS row of the O tile here and overwrites only that same row of dS later: no barrier needed in between
  row_stats_smem<HD>(p, sDO, sDS, tid, row_tok, h, Drow, lse_l2);
  const int c_lo = (row_tok / p.T) * p.T - q0, c_hi = row_last_key(p, row_tok) - q0;
  mbar_wait(&bars[1], 0);
  tc_fence_after();
  const bool uni = (p.T % 32 == 0);  // chunk window of this warp, as in the forward kernel
  bwd_softmax_tiles<true>(tS, tDP, lane_off, tid, c_lo, c_hi, p.scale * kLog2e, lse_l2, Drow, p.scale, sP, sDS,
                          attn_row_key(p, h, row_tok), q0, p.drop.thr, p.drop.scale, uni ? (c_lo >> 5) : 0, uni ? warp : 3);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
#pragma unroll
    for (int k = 0; k < kBlk / 16; ++k) {
      umma_f16(tDV, make_smem_desc(smem_u32(sP) + k * 2048, kTile, 1024), make_smem_desc(smem_u32(sDO) + k * 2048, kTile, 1024),
               idesc_g, k > 0);
    }
#pragma unroll
    for (int k = 0; k < kBlk / 16; ++k) {
      umma_f16(tDK, make_smem_desc(smem_u32(sDS) + k * 2048, kTile, 1024), make_smem_desc(smem_u32(sQ) + k * 2048, kTile, 1024),
               idesc_g, k > 0);
    }
#pragma unroll
    for (int k = 0; k < kBlk / 16; ++k) {
      umma_f16(tDQ, make_smem_desc(smem_u32(sDS) + (k >> 2) * kTile + (k & 3) * 32, 16, 1024),
               make_smem_desc(smem_u32(sK) + k * 2048, kTile, 1024), idesc_q, k > 0);
    }
    umma_commit(&bars[2]);
    }  // elect_one
  }
  mbar_wait(&bars[2], 0);
  tc_fence_after();
  // thread = token row for all three outputs (q row for dQ, key row for dK/dV).  Every MMA has completed, so the operand
  // tiles are dead: dQ / dK / dV are staged (swizzled) in the Q / K / dO tiles and leave as three TMA stores.
#pragma unroll 1
  for (int which = 0; which < 3; ++which) {
    const uint32_t t = which == 0 ? tDQ : (which == 1 ? tDK : tDV);
    uint8_t* stage = smem + which * kOp;
#pragma unroll
    for (int ch = 0; ch < HD / 32; ++ch) {
      float o[32];
      tmem_ld32(t + lane_off + ch * 32, o);
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        uint4 q;
        q.x = pack2(o[v * 8 + 0], o[v * 8 + 1]); q.y = pack2(o[v * 8 + 2], o[v * 8 + 3]);
        q.z = pack2(o[v * 8 + 4], o[v * 8 + 5]); q.w = pack2(o[v * 8 + 6], o[v * 8 + 7]);
        st_swz(stage + (ch >> 1) * kTile, tid, (ch & 1) * 4 + v, q);
      }
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  if (p.dbias) {
    // qkv bias gradient folded in: column sums of the three staged [128 x HD] tiles (the bf16 values that are stored), one
    // atomicAdd per column per CTA -- replaces a separate pass over dqkv (18 us per layer).  hd 64: thread t: tile t / 64 (and
    // the third tile split by halves), column t % 64; hd 128: column t of all three tiles.  Rows >= M were staged from zero
    // accumulators.
    const int c = tid & 63, chunk = c >> 3, within = (c & 7) * 2;
    auto colsum_rows = [&](const uint8_t* tile, int r0, int r1) {
      float acc = 0.f;
#pragma unroll 8
      for (int r = r0; r < r1; ++r)
        acc += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(tile + r * 128 + ((chunk ^ (r & 7)) << 4) + within));
      return acc;
    };
    if constexpr (HD == 64) {
      const int t01 = tid >> 6;  // 0: dQ tile, 1: dK tile
      atomicAdd(p.dbias + (t01 == 0 ? colQ : colK) + c, colsum_rows(smem + t01 * kTile, 0, kBlk));
      atomicAdd(p.dbias + colV + c, colsum_rows(smem + 2 * kTile, t01 * 64, t01 * 64 + 64));
    } else {
      const int atom = tid >> 6;  // column tid = atom tid / 64, column tid % 64 inside it
#pragma unroll 1
      for (int which = 0; which < 3; ++which)
        atomicAdd(p.dbias + (which == 0 ? colQ : (which == 1 ? colK : colV)) + tid,
                  colsum_rows(smem + which * kOp + atom * kTile, 0, kBlk));
    }
  }
  if (warp == 0) {
    if (elect_one()) {
      tma_store_tile<HD>(&p.tmap_out, smem, colQ, q0);
      tma_store_tile<HD>(&p.tmap_out, smem + kOp, colK, q0);
      tma_store_tile<HD>(&p.tmap_out, smem + 2 * kOp, colV, q0);
      tma_store_commit();
      tma_store_wait_read<0>();
    }
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem, kCols);
  }
}

}  // namespace dtb

using namespace dtb;

static void set_drop(AttnParams& p, const void* rng, int stream, float prob) {
  p.drop.rng = reinterpret_cast<const uint32_t*>(rng);
  p.drop.stream = uint32_t(stream);
  p.drop.thr = (rng && prob > 0.f) ? uint32_t(prob * 65536.f + 0.5f) : 0u;
  p.drop.scale = 1.f / (1.f - prob);
}

template <int HD>
static int attention_fwd_hd(AttnParams& p, const void* qkv, void* out, int B, int T, int H, int Hkv, int ld_qkv, int ld_out,
                            cudaStream_t s) {
  const int M = B * T;
  if (make_tmap_2d(&p.tmap_qkv, qkv, 2, uint64_t(H + 2 * Hkv) * HD, M, ld_qkv, 64, kBlk)) return 11;
  p.tmap_do = p.tmap_qkv;
  if (make_tmap_2d(&p.tmap_out, out, 2, uint64_t(H) * HD, M, ld_out, 64, kBlk)) return 11;
  static bool cfg = false;
  if (!cfg) {
    if (cudaFuncSetAttribute(attn_fwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_smem<HD>()) != cudaSuccess) return 12;
    if (cudaFuncSetAttribute(attn_fwd_small_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_small_smem<HD>()) != cudaSuccess)
      return 12;
    cfg = true;
  }
  dim3 grid((M + kBlk - 1) / kBlk, H);
  static const bool no_small = getenv("DTB200_ATTN_NO_SMALL") != nullptr;
  if (kBlk % T == 0 && !no_small) launch_pdl(attn_fwd_small_kernel<HD>, grid, dim3(128), fwd_small_smem<HD>(), s, p);  // self-contained blocks
  else attn_fwd_kernel<HD><<<grid, 128, fwd_smem<HD>(), s>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

extern "C" int dtb_attention_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, int Hkv, int hd, int ld_qkv,
                                 int ld_out, float scale, cudaStream_t s, const void* rng, int drop_stream, float drop_p,
                                 const int* kv_len) {
  if ((hd != 64 && hd != 128) || H % Hkv != 0) return 10;
  AttnParams p{};
  p.kv_len = kv_len;
  set_drop(p, rng, drop_stream, drop_p);
  p.out = (__nv_bfloat16*)out; p.lse = lse; p.M = B * T; p.T = T; p.H = H; p.Hkv = Hkv; p.ld_out = ld_out; p.ld_o = ld_out;
  p.scale = scale;
  return hd == 64 ? attention_fwd_hd<64>(p, qkv, out, B, T, H, Hkv, ld_qkv, ld_out, s)
                  : attention_fwd_hd<128>(p, qkv, out, B, T, H, Hkv, ld_qkv, ld_out, s);
}

template <int HD>
static int attention_bwd_hd(AttnParams& p, const void* dout, const void* qkv, const void* o, void* dqkv, int B, int T, int H,
                            int Hkv, int ld_qkv, int ld_o, cudaStream_t s) {
  const int M = B * T;
  if (make_tmap_2d(&p.tmap_qkv, qkv, 2, uint64_t(H + 2 * Hkv) * HD, M, ld_qkv, 64, kBlk)) return 11;
  if (make_tmap_2d(&p.tmap_do, dout, 2, uint64_t(H) * HD, M, ld_o, 64, kBlk)) return 11;
  if (make_tmap_2d(&p.tmap_o, o, 2, uint64_t(H) * HD, M, ld_o, 64, kBlk)) return 11;
  if (make_tmap_2d(&p.tmap_out, dqkv, 2, uint64_t(H + 2 * Hkv) * HD, M, ld_qkv, 64, kBlk)) return 11;
  static bool cfg = false;
  if (!cfg) {
    if (cudaFuncSetAttribute(attn_bwd_kv_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_kv_smem<HD>()) != cudaSuccess) return 12;
    if (cudaFuncSetAttribute(attn_bwd_q_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_q_smem<HD>()) != cudaSuccess) return 12;
    if (cudaFuncSetAttribute(attn_bwd_small_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_small_smem<HD>()) != cudaSuccess)
      return 12;
    cfg = true;
  }
  const int nblk = (M + kBlk - 1) / kBlk;
  static const bool no_small = getenv("DTB200_ATTN_NO_SMALL") != nullptr;
  if (p.dbias && !(kBlk % T == 0 && H == Hkv && !no_small)) return 13;  // the fold exists in the single-block kernel only
  if (kBlk % T == 0 && H == Hkv && !no_small) {
    launch_pdl(attn_bwd_small_kernel<HD>, dim3(nblk, H), dim3(128), bwd_small_smem<HD>(), s, p);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
  }
  attn_bwd_kv_kernel<HD><<<dim3(nblk, Hkv), 128, bwd_kv_smem<HD>(), s>>>(p);
  if (cudaGetLastError() != cudaSuccess) return 1;
  attn_bwd_q_kernel<HD><<<dim3(nblk, H), 128, bwd_q_smem<HD>(), s>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

extern "C" int dtb_attention_bwd(const void* dout, const void* qkv, const void* o, const float* lse, void* dqkv, int B, int T,
                                 int H, int Hkv, int hd, int ld_qkv, int ld_o, float scale, cudaStream_t s, const void* rng,
                                 int drop_stream, float drop_p, float* dbias, const int* kv_len) {
  if ((hd != 64 && hd != 128) || H % Hkv != 0) return 10;
  AttnParams p{};
  p.dbias = dbias;
  p.kv_len = kv_len;
  set_drop(p, rng, drop_stream, drop_p);
  p.o = (const __nv_bfloat16*)o; p.dout = (const __nv_bfloat16*)dout; p.out = (__nv_bfloat16*)dqkv;
  p.lse = const_cast<float*>(lse); p.M = B * T; p.T = T; p.H = H; p.Hkv = Hkv; p.ld_out = ld_qkv; p.ld_o = ld_o; p.scale = scale;
  return hd == 64 ? attention_bwd_hd<64>(p, dout, qkv, o, dqkv, B, T, H, Hkv, ld_qkv, ld_o, s)
                  : attention_bwd_hd<128>(p, dout, qkv, o, dqkv, B, T, H, Hkv, ld_qkv, ld_o, s);
}
