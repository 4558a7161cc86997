// tcgen05 GEMM / implicit-GEMM convolution for sm_100a.
//
//   out[M,N] = epilogue( A[M,K] * W[N,K]^T )           fp16 in, fp32 accumulate in TMEM, fp16 out
//
// Persistent CTAs (one per SM) walk 128 x BN output tiles. Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator
// + single thread tcgen05.mma issuer, warps 2..9 = epilogue (TMEM -> registers -> global) overlapped with the next
// tile's main loop through a double-buffered TMEM accumulator. Operands are staged by TMA into
// 128B-swizzled shared memory (64 fp16 = one 128 B row per K-block), STAGES-deep mbarrier ring.
//
// Convolution is the same kernel ("im2col-free"): the activation is NHWC, the A tile of tap (dy,dx) is a 4-D TMA box
// {64 channels, bw, bh, 1} at spatial offset (dx-1, dy-1) with out-of-bounds zero fill providing the padding; the
// weight is [Cout, taps*Cin] tap-major. Stride-2 convolutions read four parity-subsampled views of the input.
//
// Replaces (reference call sites): nn.Linear in attention_processor.py:292-320,396-453 (to_q/to_k/to_v/to_out,
// to_k_ip/to_v_ip) and, in the diffusers UNet the reference drives at custom_pipelines.py:338-345, every Linear
// (proj_in/out, FF GEGLU) and Conv2d.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdlib.h>

#include <type_traits>

#include "../../include/ih_api.h"
#include "host_util.h"
#include "ptx.cuh"

namespace ih {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KiB

struct alignas(64) TmapSet4 {
  CUtensorMap m[4];
};

struct GemmParams {
  int M, N;     // logical output rows / cols (GEGLU: N = number of gated outputs)
  int m_tiles;  // number of 128-row output tiles
  int num_kb;   // K blocks of 64 (taps * cin_kb for conv)
  int mode;     // 0 = plain GEMM, 1 = conv (4-D A maps)
  int cin_kb;   // conv: K blocks per 3x3 tap
  // conv: cumulative K-block end of every tap.  Taps 0..8 are the 3x3 window; taps 9 / 10 (optional) are a fused 1x1
  // SHORTCUT convolution over one or two further NHWC sources (ResnetBlock2D conv_shortcut on the channel concat of the
  // hidden state and the skip connection): their K blocks accumulate into the same TMEM tile, so `conv2(h) + shortcut(
  // cat(x, skip))` is ONE launch and the concatenated tensor is never materialised.
  int n_taps;
  int tap_kb_end[12];
  int Ho, Wo;   // conv: output spatial size
  int bw, bh;   // conv: spatial tile (bw*bh == 128)
  int tiles_x, tiles_y;
  signed char tap_map[12], tap_ox[12], tap_oy[12];
  int gate_row_off;  // GEGLU: row offset of the gate half inside W
  const __half* bias;
  const __half* rowbias;
  int rows_per_group;
  long long ld_rowbias;
  const __half* residual;
  long long ldr;
  __half* out;
  long long ldo;
  int act;  // 0 none, 1 SiLU, 2 GELU(erf), 3 quick-GELU (applied after bias, before residual)
  unsigned long long* trace;  // optional: %globaltimer stamps of CTA 0 (ih_gemm_set_trace), nullptr in production
  // L2 prefetch of the NEXT kernel's weights (ih_gemm_prefetch_next): inside a denoise step every GEMM streams its weights
  // from HBM (5.2 GB per step >> L2), and a launch of 5-25 us cannot hide the first HBM round trips.  An otherwise idle
  // epilogue warp issues cp.async.bulk.prefetch.L2 for this CTA's slice while the main loop runs.
  const unsigned char* pf_ptr;
  unsigned long long pf_bytes;
  int per_slab_store;   // epilogue: TMA-store every slab right after its own barrier instead of one burst per tile
  // LayerNorm folding (plain GEMM mode only).  A producer GEMM writes, per output row and 64-column slab, the sum and
  // the sum of squares of the fp16-rounded values it stores (stats_out [ceil(N/64), M, 2] fp32, one writer per slot:
  // deterministic, nothing to zero).  The consumer GEMM multiplies the RAW rows with gamma-scaled, row-CENTRED weights
  // Wc[n,k] = W[n,k] gamma[k] - mean_k(W[n,:] gamma) -- so x Wc^T = (x - mean(x)) (W gamma)^T -- and applies
  //   out = rstd[m] * acc + c[n],  c = W beta + b (passed as `bias`)   (= LayerNorm(x) W^T + b in real arithmetic)
  // with rstd rebuilt from the producer's slabs (ln_stats [ln_slabs, M, 2]).
  float alpha;   // out = alpha * acc (* rstd) + bias ...: power-of-two output scaling of the VAE's scaled residual stream
  float* stats_out;
  const float* ln_stats;
  int ln_slabs;
  float ln_inv_c;
  float ln_eps;
};

template <int BN, int STAGES, bool GEGLU, bool PAIR = false>
struct GemmSmem {
  // PAIR (cta_group::2): each CTA of the pair stages its own 128 A rows and HALF of the B tile
  static constexpr int B_STAGE_BYTES = (PAIR ? BN / 2 : BN) * BK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int TILE_BYTES = STAGES * STAGE_BYTES;
  static constexpr int BN_OUT = GEGLU ? BN / 2 : BN;
  static constexpr int SLABS = (BN_OUT + 63) / 64;   // 64-column output slabs per tile
  static constexpr int SLAB_BYTES = BM * 64 * 2;     // one 128-row x 64-column fp16 staging slab (TMA store source)
  static constexpr int BAR_BYTES = 256;
  static constexpr int BIAS_BYTES = (BN + BN_OUT) * 2;  // bias row of the tile (GEGLU: value | gate) + uniform row-bias row
  static constexpr int SMEM_LIMIT = 232448;             // 227 KiB per CTA
  // one staging slab per output slab when that fits (no buffer reuse inside a tile), else two (ping-pong)
  static constexpr int STG_SLABS =
      (TILE_BYTES + SLABS * SLAB_BYTES + BAR_BYTES + BIAS_BYTES + 1024 <= SMEM_LIMIT) ? SLABS : (SLABS < 2 ? SLABS : 2);
  static constexpr int STG_BYTES = STG_SLABS * SLAB_BYTES;
  static constexpr int BIAS_OFF = TILE_BYTES + STG_BYTES + BAR_BYTES;
  static constexpr int TOTAL = TILE_BYTES + STG_BYTES + BAR_BYTES + BIAS_BYTES + 1024;  // + alignment slack
  static_assert(TOTAL <= SMEM_LIMIT, "GEMM shared-memory budget exceeded");
  static constexpr int TMEM_COLS = 2 * BN <= 32 ? 32 : 2 * BN <= 64 ? 64 : 2 * BN <= 128 ? 128 : 2 * BN <= 256 ? 256 : 512;
};

constexpr int GEMM_EPI_WARPS = 8;
constexpr int GEMM_THREADS_P = (2 + GEMM_EPI_WARPS) * 32;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue

// Persistent kernel: grid = min(#tiles, #SMs); every CTA walks tiles blockIdx.x, +gridDim.x, ...  The smem stage
// ring runs continuously across tiles, and the fp32 accumulator is double-buffered in TMEM so that the epilogue of
// tile i (TMEM -> registers -> global, 8 warps) overlaps the TMA/MMA main loop of tile i+1.
// PAIR = true: the two CTAs of a cluster (one TPC) compute one 256 x BN tile with tcgen05.mma.cta_group::2 -- each SM
// feeds its own 128 A rows and half of B from its shared memory, which halves the per-SM operand traffic that bounds
// the single-CTA tile.  The leader CTA (cluster rank 0) issues every MMA; both CTAs run TMA producers whose loads
// complete on the leader's mbarriers; tcgen05.commit multicasts "stage free" / "accumulator ready" to both CTAs.
template <int BN, int STAGES, bool GEGLU, bool PAIR>
__global__ void __launch_bounds__(GEMM_THREADS_P, 1) gemm_f16_kernel(const __grid_constant__ TmapSet4 amaps,
                                                                      const __grid_constant__ CUtensorMap bmap,
                                                                      const __grid_constant__ CUtensorMap omap,
                                                                      const __grid_constant__ CUtensorMap rmap,
                                                                      const GemmParams p) {
  using S = GemmSmem<BN, STAGES, GEGLU, PAIR>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stg = smem + S::TILE_BYTES;            // [STG_SLABS] epilogue staging slabs, 16 KiB each (1024-aligned)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::TILE_BYTES + S::STG_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;   // [2]
  uint64_t* res_bar = tmem_empty_bar + 2;         // [4] residual slab landed (one per staging slab)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  auto stamp = [&](int slot) {
    if (p.trace && blockIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.trace[slot] = t;
    }
  };
  if (threadIdx.x == 0) stamp(0);
  constexpr int BN_OUT = GEGLU ? BN / 2 : BN;
  const int n_tiles = (p.N + BN_OUT - 1) / BN_OUT;
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = (cta_rank == 0);
  // work items: (m_unit, n_tile); an m_unit is one 128-row tile, or a pair of them (256 rows) in PAIR mode
  const int m_units = PAIR ? (p.m_tiles + 1) / 2 : p.m_tiles;
  const int num_tiles = n_tiles * m_units;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int num_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&amaps.m[0]);
    tma_prefetch_desc(&bmap);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    tma_prefetch_desc(&omap);
    for (int a = 0; a < 4; ++a) mbar_init(&res_bar[a], 1);
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], GEMM_EPI_WARPS * (PAIR ? 2 : 1));
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_2sm<S::TMEM_COLS>(tmem_slot);
    else tmem_alloc<S::TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's mbarriers must be initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) stamp(1);
  pdl_launch_dependents();  // the next kernel may begin its prologue now ...
  pdl_wait();               // ... and we may not touch global memory before our predecessor has finished
  if (threadIdx.x == 0) stamp(2);

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    // (whole warp, uniform control flow; one elected lane arms the barrier and issues the loads)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = worker; tile < num_tiles; tile += num_workers) {
        const int n_tile = tile % n_tiles;
        const int m_tile = PAIR ? 2 * (tile / n_tiles) + (int)cta_rank : tile / n_tiles;
        const int n0 = n_tile * BN_OUT;
        const int m0 = m_tile * BM;   // a dead half-tile (m_tile == m_tiles) loads zero-filled rows
        int img = 0, x0 = 0, y0 = 0;
        if (p.mode == 1) {
          const int per_img = p.tiles_x * p.tiles_y;
          img = m_tile / per_img;
          const int t = m_tile - img * per_img;
          y0 = (t / p.tiles_x) * p.bh;
          x0 = (t % p.tiles_x) * p.bw;
        }
        // conv: the tap of a K block is tracked incrementally (warp-uniform registers): tap_lo <= kb < tap_hi
        int tap = 0, tap_lo = 0, tap_hi = p.mode == 1 ? p.tap_kb_end[0] : 0x7fffffff;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          if (kb == tap_hi) {
            ++tap;
            tap_lo = tap_hi;
            tap_hi = p.tap_kb_end[tap];
          }
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sA = smem + stage * S::STAGE_BYTES;
          uint8_t* sB = sA + A_STAGE_BYTES;
          if (!elect_one()) {
            // not the issuing lane
          } else if (PAIR) {
            // both CTAs' bytes complete on the leader's barrier; only the leader arms it
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * S::STAGE_BYTES);
            if (p.mode == 0) {
              tma_load_2d_2sm(sA, &amaps.m[0], &full_bar[stage], kb * BK, m0);
            } else {
              const int ckb = kb - tap_lo;
              tma_load_4d_2sm(sA, &amaps.m[p.tap_map[tap]], &full_bar[stage], ckb * BK, x0 + p.tap_ox[tap],
                              y0 + p.tap_oy[tap], img);
            }
            // B half: leader = first BN/2 rows of the tile (GEGLU: value rows), peer = second half (GEGLU: gate rows)
            const int brow = GEGLU ? (leader ? n0 : p.gate_row_off + n0) : n0 + (int)cta_rank * (BN / 2);
            tma_load_2d_2sm(sB, &bmap, &full_bar[stage], kb * BK, brow);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], S::STAGE_BYTES);
            if (p.mode == 0) {
              tma_load_2d(sA, &amaps.m[0], &full_bar[stage], kb * BK, m0);
            } else {
              const int ckb = kb - tap_lo;
              tma_load_4d(sA, &amaps.m[p.tap_map[tap]], &full_bar[stage], ckb * BK, x0 + p.tap_ox[tap],
                          y0 + p.tap_oy[tap], img);
            }
            if (GEGLU) {
              tma_load_2d(sB, &bmap, &full_bar[stage], kb * BK, n0);
              tma_load_2d(sB + (BN / 2) * BK * 2, &bmap, &full_bar[stage], kb * BK, p.gate_row_off + n0);
            } else {
              tma_load_2d(sB, &bmap, &full_bar[stage], kb * BK, n0);
            }
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer --------------------------------
    // The whole warp walks the loop (warp-uniform control flow keeps descriptors in uniform registers); one elected
    // lane issues the MMAs and commits -- see elect_one() in ptx.cuh.
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_f16(PAIR ? 2 * BM : BM, BN, false, false);
      const uint32_t smem_lo = smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = worker; tile < num_tiles; tile += num_workers, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          if (lane == 0 && it == 0 && kb == 0) stamp(3);
          tc_fence_after();
          const uint32_t a_addr = smem_lo + stage * S::STAGE_BYTES;
          const uint64_t a_desc = umma_desc_sw128(a_addr);
          const uint64_t b_desc = umma_desc_sw128(a_addr + A_STAGE_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // +32 bytes per K=16 step inside the 128 B swizzle row (descriptor address unit = 16 B)
              if (PAIR) umma_f16_ss_2sm(tmem_d, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else umma_f16_ss(tmem_d, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            if (PAIR) umma_commit_2sm(&empty_bar[stage]);
            else umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one()) {
          if (PAIR) umma_commit_2sm(&tmem_full_bar[acc]);
          else umma_commit(&tmem_full_bar[acc]);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else {
    // ------------------------------ epilogue (8 warps, 256 threads) -------------------------------------------------
    // Latency-oriented: at UNet batch 2 most launches hold ONE tile per CTA, so the epilogue is fully exposed (trace:
    // main loop 5.6 us, old epilogue 4.6 us for a 128x192 tile against a TMEM-read floor of 0.8 us).  Therefore
    //   * the bias row of the tile (GEGLU: value | gate) and a tile-uniform row-bias row are staged in shared memory
    //     BEFORE the accumulator is ready (no dependent global loads between TMEM and the store);
    //   * every 64-column slab is drained by ALL 8 warps (warp quarter q = TMEM lanes, column half = warps 0-3 / 4-7:
    //     32 columns each), so the critical path is SLABS short steps instead of ceil(SLABS / 2) long ones;
    //   * each slab has its own staging buffer when shared memory allows (BN <= 192), else two ping-pong buffers; one
    //     thread issues all TMA loads (residual) / stores, stores are never waited for inside a tile unless a buffer
    //     is reused; residual slabs are prefetched behind the main loop.
    // TMEM -> registers (one row per thread) -> bias / LN-fold / activation / GEGLU / residual -> fp16 row segment into
    // the 128B-swizzled staging slab -> TMA store (clipped at the M / N / image edges by the tensor map).
    const int ew = warp - 2;              // 0..7
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int half = ew >> 2;             // which 32 of the 64 columns of every slab
    const int r = q * 32 + lane;          // accumulator row
    const int etid = ew * 32 + lane;      // 0..255
    const bool issuer = (ew == 0 && lane == 0);
    const int rx = r & 7;
    constexpr int SLABS = S::SLABS;
    constexpr int NBUF = S::STG_SLABS;
    __half* sBias = reinterpret_cast<__half*>(smem + S::BIAS_OFF);   // [BN]: columns of this tile (GEGLU: value | gate)
    __half* sRowb = sBias + BN;                                       // [BN_OUT]: row-bias row when uniform over the tile
    uint32_t res_par = 0;                 // bit b: parity of res_bar[b]
    if (p.pf_ptr && ew == GEMM_EPI_WARPS - 1 && lane == 0) {
      // my 1/gridDim slice of the next kernel's weights -> L2 (a hint: no completion to wait for)
      constexpr unsigned long long CH = 16384;
      const unsigned long long per = ((p.pf_bytes / gridDim.x) + CH - 1) / CH * CH;
      unsigned long long off = per * blockIdx.x;
      const unsigned long long end = off + per < p.pf_bytes ? off + per : p.pf_bytes;
      for (; off < end; off += CH) {
        const unsigned long long n = end - off < CH ? ((end - off) & ~15ull) : CH;
        if (n) l2_prefetch_bulk(p.pf_ptr + off, (uint32_t)n);
      }
    }
    int it = 0;
    for (int tile = worker; tile < num_tiles; tile += num_workers, ++it) {
      const int n_tile = tile % n_tiles;
      const int m_tile = PAIR ? 2 * (tile / n_tiles) + (int)cta_rank : tile / n_tiles;
      const int n0 = n_tile * BN_OUT;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      long long orow;
      int img = 0, x0 = 0, y0 = 0;
      const bool tile_live = m_tile < p.m_tiles;
      if (p.mode == 0) {
        orow = (long long)m_tile * BM + r;
      } else {
        const int per_img = p.tiles_x * p.tiles_y;
        img = m_tile / per_img;
        const int t = m_tile - img * per_img;
        y0 = (t / p.tiles_x) * p.bh;
        x0 = (t % p.tiles_x) * p.bw;
        const int hh = r / p.bw, ww = r - hh * p.bw;
        int y = y0 + hh, x = x0 + ww;
        if (y >= p.Ho) y = p.Ho - 1;   // clamped rows are clipped by the TMA store; keep the row-bias index in range
        if (x >= p.Wo) x = p.Wo - 1;
        orow = ((long long)img * p.Ho + y) * p.Wo + x;
      }
      const __half* rb = nullptr;
      bool rb_uniform = false;
      if (p.rowbias && tile_live) {
        const long long max_grp = ((long long)p.M - 1) / p.rows_per_group;
        long long grp = orow / p.rows_per_group;
        if (grp > max_grp) grp = max_grp;
        rb = p.rowbias + grp * p.ld_rowbias;
        if (p.mode == 1) {
          rb_uniform = true;   // a conv tile never leaves its image, rows_per_group = Ho * Wo
        } else {
          long long g0 = ((long long)m_tile * BM) / p.rows_per_group, g1 = ((long long)m_tile * BM + BM - 1) / p.rows_per_group;
          if (g1 > max_grp) g1 = max_grp;
          rb_uniform = (g0 == g1);
        }
      }
      // (a) bias rows of this tile -> shared memory (hidden behind the main loop)
      if (tile_live) {
        for (int c = etid; c < BN; c += GEMM_EPI_WARPS * 32) {
          const int lc = GEGLU ? (c < BN / 2 ? c : c - BN / 2) : c;            // tile-local output column
          const int wc = GEGLU ? (c < BN / 2 ? n0 + c : p.gate_row_off + n0 + lc) : n0 + c;   // row of W / entry of bias
          sBias[c] = (p.bias && n0 + lc < p.N) ? p.bias[wc] : __float2half_rn(0.f);
        }
        if (rb_uniform)
          for (int c = etid; c < BN_OUT; c += GEMM_EPI_WARPS * 32) sRowb[c] = (n0 + c < p.N) ? rb[n0 + c] : __float2half_rn(0.f);
      }
      // all epilogue threads: bias rows visible; the issuer has waited for the previous tile's stores (end of loop body),
      // so every staging buffer is free from here on
      named_bar_sync(1, GEMM_EPI_WARPS * 32);
      // (b) residual slabs of the first NBUF slabs are fetched now, behind the main loop
      if (issuer && tile_live && p.residual) {
        for (int sl = 0; sl < SLABS && sl < NBUF; ++sl) {
          const int col0 = n0 + sl * 64;
          if (col0 >= p.N) break;
          mbar_arrive_expect_tx(&res_bar[sl], BM * 128);
          if (p.mode == 0) tma_load_2d(stg + sl * S::SLAB_BYTES, &rmap, &res_bar[sl], col0, m_tile * BM);
          else tma_load_4d(stg + sl * S::SLAB_BYTES, &rmap, &res_bar[sl], col0, x0, y0, img);
        }
      }
      // (c) folded LayerNorm: 1 / std of my row from the producer's slabs (hidden behind the main loop of this tile)
      float ln_rstd = p.alpha;
      if (p.ln_stats && tile_live && orow < p.M) {
        const float2* st = reinterpret_cast<const float2*>(p.ln_stats) + orow;   // [slab][row]: coalesced over rows
        float ssum = 0.f, ssq = 0.f;
        for (int i0 = 0; i0 < p.ln_slabs; i0 += 10) {   // 10 independent loads in flight: one L2 round trip per 640 features
          float2 t[10];
#pragma unroll
          for (int i = 0; i < 10; ++i)
            t[i] = (i0 + i < p.ln_slabs) ? __ldg(st + (long long)(i0 + i) * p.M) : make_float2(0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 10; ++i) {
            ssum += t[i].x;
            ssq += t[i].y;
          }
        }
        const float ln_mean = ssum * p.ln_inv_c;
        const float var = fmaxf(ssq * p.ln_inv_c - ln_mean * ln_mean, 0.f);
        ln_rstd = p.alpha * rsqrtf(var + p.ln_eps);
      }

      // (d) the accumulator
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      if (threadIdx.x == 64) stamp(4 + (it < 3 ? it : 3));
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16) + half * 32;

      int last_slab = -1;
      if (tile_live)
        for (int sl = 0; sl < SLABS; ++sl)
          if (n0 + sl * 64 < p.N) last_slab = sl;
      bool arrived = false;
      // one proxy fence + barrier + store burst per tile (every slab has its own staging buffer), or store each slab as soon
      // as it is complete (p.per_slab_store: the earlier stores read their buffers out behind the later slabs' arithmetic)
      const bool kOneBarrier = (NBUF == SLABS) && !p.per_slab_store;
      // after the slab is complete in shared memory (barrier): the issuer stores it; one half-group computes the row
      // statistics of exactly the fp16 values a later LayerNorm would read -- the whole 64-column row of the slab (both
      // column halves), re-read from the staging buffer; one writer per (slab, row) slot
      auto finish_slab = [&](int sl) {
        const int col0 = n0 + sl * 64;
        uint8_t* sbuf = stg + (sl % NBUF) * S::SLAB_BYTES;
        if (issuer) {
          if (p.mode == 0) tma_store_2d(&omap, sbuf, col0, m_tile * BM);
          else tma_store_4d(&omap, sbuf, col0, x0, y0, img);
          tma_store_commit();
        }
        if (p.stats_out && half == (sl & 1) && orow < p.M) {
          const uint8_t* row_ptr = sbuf + r * 128;
          float st_sum = 0.f, st_sq = 0.f;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            if (col0 + c * 8 < p.N) {
              const uint4 o = *reinterpret_cast<const uint4*>(row_ptr + ((c ^ rx) << 4));
              const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 f = unpack_half2(ow[e]);
                st_sum += f.x + f.y;
                st_sq = fmaf(f.x, f.x, fmaf(f.y, f.y, st_sq));
              }
            }
          }
          reinterpret_cast<float2*>(p.stats_out)[(long long)(col0 >> 6) * p.M + orow] = make_float2(st_sum, st_sq);
        }
      };
      const uint32_t sbias_u32 = smem_u32(sBias);
      // arithmetic of one slab: registers (this thread's 32 accumulator columns) -> fp16 row segment in the staging slab.
      // `with_act` is a compile-time tag: the UNet's GEMMs have no activation, so they run a lean instruction stream (the
      // epilogue is latency-bound: two warps per scheduler, one dependent chain each)
      auto slab_math = [&](auto with_act, int sl, const uint32_t (&v)[32], const uint32_t (&g)[32]) {
        uint8_t* my_row = stg + (sl % NBUF) * S::SLAB_BYTES + r * 128;
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int j = half * 4 + j4;             // 16-byte chunk of the 64-column slab row
          const int lc = sl * 64 + j * 8;          // tile-local output column of the chunk
          float x[8];
          {
            // acc * rstd + bias: rstd = alpha without a folded LayerNorm; with one, `bias` carries W beta + b and the
            // weight rows are gamma-scaled AND centred, so the mean term has already cancelled inside the MMA
            const uint4 bv = lds128(sbias_u32 + lc * 2);
            const uint32_t bw[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = unpack_half2(bw[e]);
              x[2 * e] = fmaf(ln_rstd, __uint_as_float(v[j4 * 8 + 2 * e]), f.x);
              x[2 * e + 1] = fmaf(ln_rstd, __uint_as_float(v[j4 * 8 + 2 * e + 1]), f.y);
            }
          }
          if (GEGLU) {
            float gt[8];
            const uint4 gv = lds128(sbias_u32 + (BN / 2 + lc) * 2);
            const uint32_t bw[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = unpack_half2(bw[e]);
              gt[2 * e] = fmaf(ln_rstd, __uint_as_float(g[j4 * 8 + 2 * e]), f.x);
              gt[2 * e + 1] = fmaf(ln_rstd, __uint_as_float(g[j4 * 8 + 2 * e + 1]), f.y);
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) x[e] *= gelu_erf_f(gt[e]);
          }
          if (rb) {
            uint4 rv;
            if (rb_uniform) {
              rv = lds128(sbias_u32 + (BN + lc) * 2);
            } else {   // rows of several groups in one tile (not used by the UNet): per-row global loads
              int col = n0 + lc;
              if (col > p.N - 8) col = p.N - 8;
              rv = __ldg(reinterpret_cast<const uint4*>(rb + col));
            }
            const uint32_t bw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = unpack_half2(bw[e]);
              x[2 * e] += f.x;
              x[2 * e + 1] += f.y;
            }
          }
          if constexpr (decltype(with_act)::value) {
            if (p.act == 1) {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = silu_f(x[e]);
            } else if (p.act == 2) {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = gelu_erf_f(x[e]);
            } else if (p.act == 3) {   // quick_gelu x * sigmoid(1.702 x) ([3P] CLIP-L text tower MLP)
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = __fdividef(x[e], 1.f + __expf(-1.702f * x[e]));
            }
          }
          uint4* slot = reinterpret_cast<uint4*>(my_row + ((j ^ rx) << 4));
          if (p.residual) {
            const uint4 b4 = *slot;
            const uint32_t bw[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = unpack_half2(bw[e]);
              x[2 * e] += f.x;
              x[2 * e + 1] += f.y;
            }
          }
          uint4 o;
          o.x = pack_half2(x[0], x[1]);
          o.y = pack_half2(x[2], x[3]);
          o.z = pack_half2(x[4], x[5]);
          o.w = pack_half2(x[6], x[7]);
          *slot = o;
        }
      };
      // staging-buffer reuse (BN = 256 without GEGLU only): the store of slab sl - NBUF must have read the buffer out; then
      // the residual slab is fetched into it
      auto reuse_buffer = [&](int sl) {
        const int col0 = n0 + sl * 64;
        const int buf = sl % NBUF;
        uint8_t* sbuf = stg + buf * S::SLAB_BYTES;
        if (issuer) {
          tma_store_wait_read<(NBUF > 1 ? NBUF - 1 : 0)>();
          if (p.residual) {
            mbar_arrive_expect_tx(&res_bar[buf], BM * 128);
            if (p.mode == 0) tma_load_2d(sbuf, &rmap, &res_bar[buf], col0, m_tile * BM);
            else tma_load_4d(sbuf, &rmap, &res_bar[buf], col0, x0, y0, img);
          }
        }
        named_bar_sync(2, GEMM_EPI_WARPS * 32);
      };
      auto release_accumulator = [&]() {
        // this warp's last TMEM read of the accumulator is complete: hand the buffer back to the MMA warp
        arrived = true;
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR && !leader) mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty_bar[acc]), 0));
          else mbar_arrive(&tmem_empty_bar[acc]);
        }
      };
      auto wait_residual = [&](int sl) {
        if (p.residual) {
          const int buf = sl % NBUF;
          mbar_wait(&res_bar[buf], (res_par >> buf) & 1u);
          res_par ^= 1u << buf;
        }
      };
      auto slab_done = [&](int sl) {
        if (issuer && it == 0 && sl == 0) stamp(10);
        if (!kOneBarrier) {
          fence_proxy_async_smem();
          named_bar_sync(3, GEMM_EPI_WARPS * 32);      // the slab is complete in shared memory
          if (issuer && it == 0) stamp(sl == last_slab ? 12 : 11);
          finish_slab(sl);
        }
      };
      if (!GEGLU && p.act == 0) {
        // fast path (every GEMM / conv of the UNet except the FF GEGLU-in): no activation code, and the TMEM load of
        // slab sl + 1 is in flight during the arithmetic of slab sl (two register buffers)
        uint32_t v[2][32];
        if (last_slab >= 0) tmem_ld_32x32b_x32(taddr, v[0]);
#pragma unroll
        for (int sl = 0; sl < SLABS; ++sl) {
          if (sl <= last_slab) {
            if (sl >= NBUF) reuse_buffer(sl);
            tmem_ld_wait();
            if (issuer && it == 0 && sl == 0) stamp(9);
            if (sl + 1 < SLABS && sl + 1 <= last_slab) tmem_ld_32x32b_x32(taddr + (sl + 1) * 64, v[(sl + 1) & 1]);
            if (sl == last_slab) release_accumulator();
            wait_residual(sl);
            slab_math(std::false_type{}, sl, v[sl & 1], v[sl & 1]);
            slab_done(sl);
          }
        }
      } else {
#pragma unroll 1
        for (int sl = 0; sl <= last_slab; ++sl) {
          uint32_t v[32];
          uint32_t g[32];
          tmem_ld_32x32b_x32(taddr + sl * 64, v);
          if (GEGLU) tmem_ld_32x32b_x32(taddr + BN / 2 + sl * 64, g);
          if (sl >= NBUF) reuse_buffer(sl);
          tmem_ld_wait();
          if (issuer && it == 0 && sl == 0) stamp(9);
          if (sl == last_slab) release_accumulator();
          wait_residual(sl);
          slab_math(std::true_type{}, sl, v, g);
          slab_done(sl);
        }
      }
      if (kOneBarrier && last_slab >= 0) {
        // every slab has its own staging buffer: ONE proxy fence + ONE barrier for the whole tile, then all stores
        fence_proxy_async_smem();
        named_bar_sync(3, GEMM_EPI_WARPS * 32);
        if (issuer && it == 0) stamp(12);
        for (int sl = 0; sl <= last_slab; ++sl) finish_slab(sl);
      }
      if (!arrived) {   // no live slab in the tile (dead half tile of a CTA pair): still release the accumulator
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR && !leader) mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty_bar[acc]), 0));
          else mbar_arrive(&tmem_empty_bar[acc]);
        }
      }
      // the staging buffers may be rewritten (next tile) / must stay valid (kernel end) until the bulk stores have read
      // them; global visibility is given by kernel completion (the next kernel's griddepcontrol.wait / stream order)
      if (issuer) tma_store_wait_read0();
      if (issuer && it == 0) stamp(13);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) stamp(8);
  if (PAIR) cluster_sync_all();   // nobody may exit (or free TMEM) while the peer can still signal / read it
  if (warp == 1) {
    if (PAIR) tmem_dealloc_2sm<S::TMEM_COLS>(tmem_base);
    else tmem_dealloc<S::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
template <int BN, int STAGES, bool GEGLU, bool PAIR = false>
static int launch_gemm(const TmapSet4& amaps, const CUtensorMap& bmap, const CUtensorMap& omap,
                       const CUtensorMap& rmap, GemmParams& p, int m_tiles, cudaStream_t stream) {
  using S = GemmSmem<BN, STAGES, GEGLU, PAIR>;
  static bool configured = false;
  auto kern = gemm_f16_kernel<BN, STAGES, GEGLU, PAIR>;
  if (!configured) {
    IH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    configured = true;
  }
  constexpr int BN_OUT = GEGLU ? BN / 2 : BN;
  p.m_tiles = m_tiles;
  const long long n_tiles = (p.N + BN_OUT - 1) / BN_OUT;
  if (PAIR) {
    const long long units = n_tiles * ((m_tiles + 1) / 2);
    const long long pairs = num_sms() / 2;
    const int grid = 2 * (int)(units < pairs ? units : pairs);
    IH_CUDA(launch_kernel_cluster(kern, dim3(grid), dim3(GEMM_THREADS_P), (size_t)(S::TOTAL), stream, 2, amaps, bmap, omap, rmap, p));
    return 0;
  }
  const long long tiles = n_tiles * m_tiles;
  const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
  IH_CUDA(launch_kernel(kern, dim3(grid), dim3(GEMM_THREADS_P), (size_t)(S::TOTAL), stream, amaps, bmap, omap, rmap, p));
  return 0;
}

// Cost model for the persistent kernel (one CTA per SM), calibrated on B200 (tools/microbench.py):
//   * a 128x256 tile streams 48 KiB of operands per 2^22 MACs; a 128x128 tile 32 KiB per 2^21 MACs -- the narrower
//     tile needs 1.33x the L2->SM bytes per FLOP and is latency/L2-bound (785 vs 1180 TFLOP/s at 8192^3), so its cost
//     per tile is ~0.75 of the wide tile, not 0.5; 128x64 tiles are worse still and only used for N <= 64.
//   * padded columns of a partially filled last N tile cost as much as real ones.
static int pick_bn(long long m_tiles, int N) {
  if (N <= 64) return 64;
  const int sms = num_sms();
  double best = 1e30;
  int best_bn = 256;
  // 128x64 tiles for launches that cannot fill the SMs with wider ones (the 1280-channel level of a 512^2 edit has
  // M = 512: 28 tiles of 128x192): each SM then streams 24 instead of 32-40 KB per k-block and drains one slab.
  // Same-box A/B: 512^2 step 10.47 -> 9.84 ms (GEMMs) -> 9.76 ms (+ convs), 1024^2 unchanged.  IH_BN64=0 disables.
  static const int bn64 = [] {
    const char* e = getenv("IH_BN64");
    return e ? atoi(e) : 1;
  }();
  if (bn64 && m_tiles * ((N + 63) / 64) <= sms) return 64;
  // per-tile main-loop cost relative to the 128x256 tile.  Measured per 64-deep k-block with 144 CTAs busy
  // (tools/ab_probe.py tile): 0.350 us (256), 0.276 us (192), 0.257 us (128) -- the narrow tiles move more operand
  // bytes per FLOP and the main loop is bound by the L2 -> SM operand stream (~19 TB/s aggregate), not by the MMA.
  const int cands[3] = {256, 192, 128};
  const double tile_cost[3] = {2.0, 1.58, 1.47};
  for (int i = 0; i < 3; ++i) {
    const int bn = cands[i];
    const long long tiles = m_tiles * ((N + bn - 1) / bn);
    const long long rounds = (tiles + sms - 1) / sms;
    const double t = (double)rounds * (tile_cost[i] + 0.15);
    if (t < best - 1e-9) {
      best = t;
      best_bn = bn;
    }
  }
  return best_bn;
}

// IH_GEMM_PAIR: 0 = never use the CTA-pair tile, 1 = cost model (default), 2 = whenever N >= 256
static int pair_mode() {
  static int m = [] {
    const char* e = getenv("IH_GEMM_PAIR");
    return e ? atoi(e) : 1;
  }();
  return m;
}
// Measured on B200 (tools/overhead_probe.py, tools/microbench.py): a cluster launch + two cluster barriers cost ~5 us
// more than a plain launch (10.7 vs 5.7 us for a one-tile GEMM) while the pair main loop is only ~5 % faster than
// the single-CTA 128x256 tile, so the pair tile pays off only for long-running GEMMs.
static bool pair_is_faster(long long m_tiles, int n_cols, int num_kb) {
  const int sms = num_sms();
  const long long nt = (n_cols + 255) / 256;
  const long long r1 = (m_tiles * nt + sms - 1) / sms;                       // single-CTA 128x256 tiles
  const long long r2 = (((m_tiles + 1) / 2) * nt + sms / 2 - 1) / (sms / 2);  // pair 256x256 tiles
  const double kb_us = 0.30;
  const double t1 = (double)r1 * num_kb * kb_us + 5.7, t2 = (double)r2 * num_kb * kb_us / 1.05 + 10.7;
  return t2 < t1;
}

static int dispatch(const TmapSet4& amaps, const CUtensorMap& omap, const CUtensorMap& rmap, const void* w, int ldw_rows,
                    long long K, GemmParams& p, int m_tiles, int geglu, int force_bn, cudaStream_t stream) {
  // tile_n = 512 forces the CTA-pair 256x256 tile, 384 the CTA-pair 256x192 tile, other explicit values force the
  // single-CTA tile of that width
  bool pair = false;
  // CTA-pair 256x192 tile: the same tiles per SM as the single-CTA 128x192 tile, but every SM streams half of B (28
  // instead of 40 KB per k-block).  The main loop is bound by the L2 -> SM operand stream, so long-K launches gain
  // (tools/tile_probe.py, profiles/r2_tile_probe.txt: conv3x3 2560->1280 118 -> 95 us, 1280->1280 53 -> 50 us, FF-out
  // K = 5120 27.5 -> 26.2 us) while the ~0.5 us of cluster set-up loses on K = 1280 (11.1 -> 11.5 us): used from 40
  // k-blocks on.  IH_PAIR192=0 disables the heuristic.
  static const bool pair192_on = [] {
    const char* e = getenv("IH_PAIR192");
    return !(e && e[0] == '0');
  }();
  static const int pair192_min_kb = [] {
    const char* e = getenv("IH_PAIR192_MINKB");
    return e ? atoi(e) : 40;
  }();
  const bool want_pair192 = force_bn == 384 || (force_bn == 0 && pair192_on && !geglu && p.num_kb >= pair192_min_kb && m_tiles >= 2 &&
                                                 p.N > 64 && pick_bn(m_tiles, p.N) == 192 &&
                                                 !(pair_mode() != 0 && p.N >= 256 && pair_is_faster(m_tiles, p.N, p.num_kb)));
  if (want_pair192 && !geglu) {
    CUtensorMap bmap192;
    const uint64_t bdims[2] = {(uint64_t)K, (uint64_t)ldw_rows};
    const uint64_t bstr[1] = {(uint64_t)K * 2};
    const uint32_t bbox[2] = {(uint32_t)BK, 96u};
    int rc = get_tmap_f16(&bmap192, w, 2, bdims, bstr, bbox);
    if (rc) return rc;
    return launch_gemm<192, 6, false, true>(amaps, bmap192, omap, rmap, p, m_tiles, stream);
  }
  if (force_bn == 512) {
    pair = true;
    force_bn = 256;
  } else if (force_bn == 0 && pair_mode() != 0 && (geglu || p.N >= 256)) {
    // GEGLU on CTA-pair tiles from 20 k-blocks on: measured in the step (tools/ab_env.sh, two repeats on one box) 19.23 ->
    // 19.10 ms for the 2048 x 10240 x 1280 FF GEGLU-in (micro-benchmark 44.3 -> 41.4 us), while the K = 640 level loses
    // (52.3 -> 59.0 us).  IH_GEGLU_PAIR=0 / 1 overrides (never / always).
    static const int geglu_pair = [] {
      const char* e = getenv("IH_GEGLU_PAIR");
      return e ? (e[0] == '1' ? 1 : 0) : -1;
    }();
    const bool geglu_wants_pair = geglu && (geglu_pair == 1 || (geglu_pair == -1 && p.num_kb >= 20));
    pair = pair_mode() == 2 || geglu_wants_pair || pair_is_faster(m_tiles, geglu ? 2 * p.N : p.N, p.num_kb);
  }
  int bn = (geglu || pair) ? 256 : (force_bn > 0 ? force_bn : pick_bn(m_tiles, p.N));
  CUtensorMap bmap;
  const uint64_t bdims[2] = {(uint64_t)K, (uint64_t)ldw_rows};
  const uint64_t bstr[1] = {(uint64_t)K * 2};
  const uint32_t bbox[2] = {(uint32_t)BK, (uint32_t)((geglu || pair) ? 128 : bn)};
  int rc = get_tmap_f16(&bmap, w, 2, bdims, bstr, bbox);
  if (rc) return rc;
  if (pair) {
    if (geglu) return launch_gemm<256, 6, true, true>(amaps, bmap, omap, rmap, p, m_tiles, stream);
    return launch_gemm<256, 6, false, true>(amaps, bmap, omap, rmap, p, m_tiles, stream);
  }
  if (geglu) return launch_gemm<256, 4, true>(amaps, bmap, omap, rmap, p, m_tiles, stream);
  switch (bn) {
    case 256: return launch_gemm<256, 4, false>(amaps, bmap, omap, rmap, p, m_tiles, stream);
    case 192: return launch_gemm<192, 4, false>(amaps, bmap, omap, rmap, p, m_tiles, stream);
    case 128: return launch_gemm<128, 6, false>(amaps, bmap, omap, rmap, p, m_tiles, stream);
    case 64: return launch_gemm<64, 8, false>(amaps, bmap, omap, rmap, p, m_tiles, stream);
    default: return set_error(IH_ERR_ARG, "unsupported BN %d", bn);
  }
}

// IH_EPI_PER_SLAB=1: per-slab TMA stores in the epilogue (A/B switch; default: one store burst per tile)
static int per_slab_store_mode() {
  static int m = [] {
    const char* e = getenv("IH_EPI_PER_SLAB");
    return (e && e[0] == '1') ? 1 : 0;
  }();
  return m;
}
static unsigned long long* g_trace = nullptr;
// one-shot hint consumed by the next GEMM / conv launch of this thread (ih_gemm_prefetch_next)
static thread_local const void* g_pf_ptr = nullptr;
static thread_local unsigned long long g_pf_bytes = 0;
// The hint is consumed by the FIRST launch attempt after it was set, whether or not that call gets as far as launching:
// a call that fails validation must not leave a pointer behind for an unrelated later launch.
struct PrefetchHint {
  const unsigned char* ptr;
  unsigned long long bytes;
};
static PrefetchHint take_prefetch_hint() {
  PrefetchHint h{(const unsigned char*)g_pf_ptr, g_pf_bytes};
  g_pf_ptr = nullptr;
  g_pf_bytes = 0;
  return h;
}
}  // namespace ih

using namespace ih;

// debugging aid: device buffer of >= 16 uint64 that CTA 0 of subsequent GEMM launches fills with %globaltimer stamps
// (0 kernel entry, 1 setup done, 2 predecessor finished, 3 first operands landed, 4..7 accumulator ready for tiles
// 0..3+, 8 CTA done); pass NULL to disable.
extern "C" void ih_gemm_set_trace(void* device_buffer) { ih::g_trace = (unsigned long long*)device_buffer; }

extern "C" void ih_gemm_prefetch_next(const void* weights, long long bytes) {
  ih::g_pf_ptr = (weights && bytes >= 16 && ((uintptr_t)weights & 15) == 0) ? weights : nullptr;
  ih::g_pf_bytes = ih::g_pf_ptr ? (unsigned long long)bytes : 0;
}

static int gemm_impl(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                     int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                     long long ldo, int M, int N, int K, int epilogue, int tile_n, const void* ln_stats,
                     int ln_slabs, float ln_eps, void* stats_out, float alpha, void* stream);

extern "C" int ih_gemm_f16(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                           int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                           long long ldo, int M, int N, int K, int epilogue, int tile_n, void* stream) {
  return gemm_impl(a, lda, w, bias, rowbias, rows_per_group, ld_rowbias, residual, ldr, out, ldo, M, N, K, epilogue,
                   tile_n, nullptr, 0, 0.f, nullptr, 1.f, stream);
}

extern "C" int ih_gemm_scaled_f16(const void* a, long long lda, const void* w, const void* bias, const void* residual,
                                  long long ldr, void* out, long long ldo, int M, int N, int K, int epilogue, float alpha,
                                  void* stream) {
  return gemm_impl(a, lda, w, bias, nullptr, 0, 0, residual, ldr, out, ldo, M, N, K, epilogue, 0, nullptr, 0, 0.f,
                   nullptr, alpha, stream);
}

extern "C" int ih_gemm_ln_f16(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                              int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                              long long ldo, int M, int N, int K, int epilogue, int tile_n, const void* ln_stats,
                              int ln_slabs, float ln_eps, void* stats_out, void* stream) {
  return gemm_impl(a, lda, w, bias, rowbias, rows_per_group, ld_rowbias, residual, ldr, out, ldo, M, N, K, epilogue,
                   tile_n, ln_stats, ln_slabs, ln_eps, stats_out, 1.f, stream);
}

static int gemm_impl(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                     int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                     long long ldo, int M, int N, int K, int epilogue, int tile_n, const void* ln_stats,
                     int ln_slabs, float ln_eps, void* stats_out, float alpha, void* stream) {
  const PrefetchHint hint = take_prefetch_hint();
  IH_CHECK(a && w && out, IH_ERR_ARG, "ih_gemm_f16: null pointer");
  IH_CHECK(M > 0 && N > 0 && K > 0, IH_ERR_SHAPE, "ih_gemm_f16: bad shape M=%d N=%d K=%d", M, N, K);
  IH_CHECK(K % 8 == 0 && N % 8 == 0 && lda % 8 == 0 && ldo % 8 == 0, IH_ERR_ALIGN,
           "ih_gemm_f16: K, N, lda, ldo must be multiples of 8 (16-byte rows)");
  const bool geglu = (epilogue & IH_EPI_GEGLU) != 0;
  IH_CHECK(!geglu || (N % 16 == 0), IH_ERR_SHAPE, "ih_gemm_f16: GEGLU needs even split of N");
  IH_CHECK(!(residual) || ldr % 8 == 0, IH_ERR_ALIGN, "ih_gemm_f16: ldr must be a multiple of 8");
  IH_CHECK(!rowbias || (rows_per_group > 0 && ld_rowbias % 8 == 0), IH_ERR_ARG,
           "ih_gemm_f16: rowbias needs rows_per_group > 0 and ld_rowbias %% 8 == 0");

  TmapSet4 amaps;
  const uint64_t adims[2] = {(uint64_t)K, (uint64_t)M};
  const uint64_t astr[1] = {(uint64_t)lda * 2};
  const uint32_t abox[2] = {(uint32_t)BK, (uint32_t)BM};
  int rc = get_tmap_f16(&amaps.m[0], a, 2, adims, astr, abox);
  if (rc) return rc;
  amaps.m[1] = amaps.m[2] = amaps.m[3] = amaps.m[0];

  GemmParams p{};
  p.M = M;
  p.N = geglu ? N / 2 : N;
  p.num_kb = (K + BK - 1) / BK;
  p.mode = 0;
  p.gate_row_off = geglu ? N / 2 : 0;
  p.bias = (const __half*)bias;
  p.rowbias = (const __half*)rowbias;
  p.rows_per_group = rows_per_group > 0 ? rows_per_group : 1;
  p.ld_rowbias = ld_rowbias;
  p.residual = (const __half*)residual;
  p.ldr = ldr;
  p.out = (__half*)out;
  p.ldo = ldo;
  p.act = (epilogue & IH_EPI_SILU) ? 1 : ((epilogue & IH_EPI_GELU) ? 2 : ((epilogue & IH_EPI_QUICK_GELU) ? 3 : 0));
  p.trace = g_trace;
  p.pf_ptr = hint.ptr;
  p.pf_bytes = hint.bytes;
  p.per_slab_store = per_slab_store_mode();
  IH_CHECK(!ln_stats || ln_slabs > 0, IH_ERR_ARG, "ih_gemm_ln_f16: ln_stats needs ln_slabs > 0");
  IH_CHECK(!stats_out || N % 64 == 0 || geglu, IH_ERR_SHAPE, "ih_gemm_ln_f16: stats_out needs N %% 64 == 0");
  p.stats_out = (float*)stats_out;
  p.ln_stats = (const float*)ln_stats;
  p.ln_slabs = ln_slabs;
  p.ln_inv_c = 1.0f / (float)K;
  p.ln_eps = ln_eps;
  p.alpha = alpha;
  const int m_tiles = (M + BM - 1) / BM;
  CUtensorMap omap, rmap;
  {
    const uint64_t odims[2] = {(uint64_t)p.N, (uint64_t)M};
    const uint32_t obox[2] = {64u, (uint32_t)BM};
    const uint64_t ostr[1] = {(uint64_t)ldo * 2};
    rc = get_tmap_f16(&omap, out, 2, odims, ostr, obox);
    if (rc) return rc;
    rmap = omap;
    if (residual) {
      const uint64_t rstr[1] = {(uint64_t)ldr * 2};
      rc = get_tmap_f16(&rmap, residual, 2, odims, rstr, obox);
      if (rc) return rc;
    }
  }
  return dispatch(amaps, omap, rmap, w, N, K, p, m_tiles, geglu, tile_n, (cudaStream_t)stream);
}

static int conv_impl(const void* x, const void* w, const void* bias, const void* rowbias, long long ld_rowbias,
                     const void* residual, void* out, int B, int Hin, int Win, int Cin, int Cout, int ksize, int stride,
                     int tile_n, float alpha, void* stream, const void* sc0 = nullptr, int Csc0 = 0,
                     const void* sc1 = nullptr, int Csc1 = 0, bool pad_br = false);

extern "C" int ih_conv2d_f16(const void* x, const void* w, const void* bias, const void* rowbias,
                             long long ld_rowbias, const void* residual, void* out, int B, int Hin, int Win, int Cin,
                             int Cout, int ksize, int stride, int tile_n, void* stream) {
  return conv_impl(x, w, bias, rowbias, ld_rowbias, residual, out, B, Hin, Win, Cin, Cout, ksize, stride, tile_n, 1.f,
                   stream);
}

extern "C" int ih_conv2d_scaled_f16(const void* x, const void* w, const void* bias, const void* residual, void* out,
                                    int B, int Hin, int Win, int Cin, int Cout, int stride, float alpha, void* stream) {
  return conv_impl(x, w, bias, nullptr, 0, residual, out, B, Hin, Win, Cin, Cout, 3, stride, 0, alpha, stream);
}

extern "C" int ih_conv2d_s2_padbr_f16(const void* x, const void* w, const void* bias, void* out, int B, int Hin, int Win,
                                      int Cin, int Cout, void* stream) {
  return conv_impl(x, w, bias, nullptr, 0, nullptr, out, B, Hin, Win, Cin, Cout, 3, 2, 0, 1.f, stream, nullptr, 0, nullptr,
                   0, true);
}

extern "C" int ih_conv2d_shortcut_f16(const void* x, const void* w, const void* bias, const void* rowbias,
                                      long long ld_rowbias, const void* sc0, int Csc0, const void* sc1, int Csc1, void* out,
                                      int B, int H, int W, int Cin, int Cout, void* stream) {
  IH_CHECK(sc0 && Csc0 > 0 && Csc0 % BK == 0 && (!sc1 || (Csc1 > 0 && Csc1 % BK == 0)), IH_ERR_SHAPE,
           "ih_conv2d_shortcut_f16: shortcut sources need channel counts that are multiples of 64");
  return conv_impl(x, w, bias, rowbias, ld_rowbias, nullptr, out, B, H, W, Cin, Cout, 3, 1, 0, 1.f, stream, sc0, Csc0,
                   sc1 ? sc1 : nullptr, sc1 ? Csc1 : 0);
}

static int conv_impl(const void* x, const void* w, const void* bias, const void* rowbias, long long ld_rowbias,
                     const void* residual, void* out, int B, int Hin, int Win, int Cin, int Cout, int ksize, int stride,
                     int tile_n, float alpha, void* stream, const void* sc0, int Csc0, const void* sc1, int Csc1,
                     bool pad_br) {
  const PrefetchHint hint = take_prefetch_hint();
  IH_CHECK(x && w && out, IH_ERR_ARG, "ih_conv2d_f16: null pointer");
  IH_CHECK(ksize == 3, IH_ERR_ARG, "ih_conv2d_f16: ksize must be 3 (1x1 convs are ih_gemm_f16)");
  IH_CHECK(stride == 1 || stride == 2, IH_ERR_ARG, "ih_conv2d_f16: stride must be 1 or 2");
  IH_CHECK(Cin % 8 == 0 && Cout % 8 == 0, IH_ERR_ALIGN, "ih_conv2d_f16: channels must be multiples of 8");
  IH_CHECK(stride == 1 || (Hin % 2 == 0 && Win % 2 == 0), IH_ERR_SHAPE, "ih_conv2d_f16: stride 2 needs even H, W");
  const int Ho = Hin / stride, Wo = Win / stride;

  // spatial tile: bw x bh = 128 output pixels, minimise padded tiles
  int best_bw = 128;
  long long best_tiles = -1;
  for (int bw = 128; bw >= 1; bw >>= 1) {
    const int bh = 128 / bw;
    const long long t = (long long)((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh);
    if (best_tiles < 0 || t < best_tiles) {
      best_tiles = t;
      best_bw = bw;
    }
  }
  GemmParams p{};
  p.bw = best_bw;
  p.bh = 128 / best_bw;
  p.tiles_x = (Wo + p.bw - 1) / p.bw;
  p.tiles_y = (Ho + p.bh - 1) / p.bh;
  p.Ho = Ho;
  p.Wo = Wo;
  p.mode = 1;
  p.cin_kb = (Cin + BK - 1) / BK;
  p.n_taps = 9;
  for (int t = 0; t < 9; ++t) p.tap_kb_end[t] = (t + 1) * p.cin_kb;
  if (sc0) {
    p.tap_kb_end[9] = p.tap_kb_end[8] + Csc0 / BK;
    p.n_taps = 10;
    if (sc1) {
      p.tap_kb_end[10] = p.tap_kb_end[9] + Csc1 / BK;
      p.n_taps = 11;
    }
  }
  for (int t = p.n_taps; t < 12; ++t) p.tap_kb_end[t] = 0x7fffffff;   // sentinel: the tap search always terminates
  p.num_kb = p.tap_kb_end[p.n_taps - 1];
  p.M = B * Ho * Wo;
  p.N = Cout;
  p.bias = (const __half*)bias;
  p.rowbias = (const __half*)rowbias;
  p.rows_per_group = Ho * Wo;
  p.ld_rowbias = ld_rowbias;
  p.residual = (const __half*)residual;
  p.ldr = Cout;
  p.out = (__half*)out;
  p.ldo = Cout;
  p.trace = g_trace;
  p.pf_ptr = hint.ptr;
  p.pf_bytes = hint.bytes;
  p.per_slab_store = per_slab_store_mode();
  p.alpha = alpha;

  TmapSet4 amaps;
  const uint32_t abox[4] = {(uint32_t)BK, (uint32_t)p.bw, (uint32_t)p.bh, 1u};
  if (stride == 1) {
    const uint64_t adims[4] = {(uint64_t)Cin, (uint64_t)Win, (uint64_t)Hin, (uint64_t)B};
    const uint64_t astr[3] = {(uint64_t)Cin * 2, (uint64_t)Win * Cin * 2, (uint64_t)Hin * Win * Cin * 2};
    int rc = get_tmap_f16(&amaps.m[0], x, 4, adims, astr, abox);
    if (rc) return rc;
    amaps.m[1] = amaps.m[2] = amaps.m[3] = amaps.m[0];
    for (int t = 0; t < 9; ++t) {
      p.tap_map[t] = 0;
      p.tap_ox[t] = (signed char)(t % 3 - 1);
      p.tap_oy[t] = (signed char)(t / 3 - 1);
    }
    const void* srcs[2] = {sc0, sc1};
    const int chans[2] = {Csc0, Csc1};
    for (int i = 0; i < 2 && srcs[i]; ++i) {       // fused 1x1 shortcut sources: centre tap of their own tensor maps
      const uint64_t sdims[4] = {(uint64_t)chans[i], (uint64_t)Win, (uint64_t)Hin, (uint64_t)B};
      const uint64_t sstr[3] = {(uint64_t)chans[i] * 2, (uint64_t)Win * chans[i] * 2, (uint64_t)Hin * Win * chans[i] * 2};
      rc = get_tmap_f16(&amaps.m[1 + i], srcs[i], 4, sdims, sstr, abox);
      if (rc) return rc;
      p.tap_map[9 + i] = (signed char)(1 + i);
      p.tap_ox[9 + i] = p.tap_oy[9 + i] = 0;
    }
  } else {
    IH_CHECK(!sc0, IH_ERR_ARG, "ih_conv2d: a fused shortcut needs stride 1");
    // padding 1: input row 2*oy + dy - 1: dy=0 -> odd rows at oy-1, dy=1 -> even rows at oy, dy=2 -> odd rows at oy.
    // pad_br (bottom / right padding only): input row 2*oy + dy: dy=0 -> even rows at oy, dy=1 -> odd rows at oy,
    // dy=2 -> even rows at oy+1, which is out of bounds on the last output row and column: TMA fills it with zeros.
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        const __half* base = (const __half*)x + ((long long)py * Win + px) * Cin;
        const uint64_t adims[4] = {(uint64_t)Cin, (uint64_t)Win / 2, (uint64_t)Hin / 2, (uint64_t)B};
        const uint64_t astr[3] = {(uint64_t)2 * Cin * 2, (uint64_t)2 * Win * Cin * 2, (uint64_t)Hin * Win * Cin * 2};
        int rc = get_tmap_f16(&amaps.m[py * 2 + px], base, 4, adims, astr, abox);
        if (rc) return rc;
      }
    const int par[3] = {pad_br ? 0 : 1, pad_br ? 1 : 0, pad_br ? 0 : 1};
    const int off[3] = {pad_br ? 0 : -1, 0, pad_br ? 1 : 0};
    for (int t = 0; t < 9; ++t) {
      const int dy = t / 3, dx = t % 3;
      p.tap_map[t] = (signed char)(par[dy] * 2 + par[dx]);
      p.tap_ox[t] = (signed char)off[dx];
      p.tap_oy[t] = (signed char)off[dy];
    }
  }
  const int m_tiles = B * p.tiles_x * p.tiles_y;
  // weight is [Cout, 9*Cin] tap-major; when Cin is not a multiple of 64 each tap's K range is padded by TMA zero fill
  IH_CHECK(Cin % BK == 0, IH_ERR_SHAPE, "ih_conv2d_f16: Cin must be a multiple of 64 (got %d)", Cin);
  CUtensorMap omap, rmap;
  {
    const uint64_t odims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)B};
    const uint64_t ostr[3] = {(uint64_t)Cout * 2, (uint64_t)Wo * Cout * 2, (uint64_t)Ho * Wo * Cout * 2};
    const uint32_t obox[4] = {64u, (uint32_t)p.bw, (uint32_t)p.bh, 1u};
    int rc = get_tmap_f16(&omap, out, 4, odims, ostr, obox);
    if (rc) return rc;
    rmap = omap;
    if (residual) {
      rc = get_tmap_f16(&rmap, residual, 4, odims, ostr, obox);
      if (rc) return rc;
    }
  }
  return dispatch(amaps, omap, rmap, w, Cout, (long long)9 * Cin + Csc0 + Csc1, p, m_tiles, 0, tile_n, (cudaStream_t)stream);
}
