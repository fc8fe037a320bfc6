// K1: grouped, expert-bucketed GEMM / implicit-GEMM 3x3 conv for sm_100a.
//
//   out[row, n] = epilogue( sum_{tap, c} A[pixel(row) + tap, c] * W[w_row_off + n, tap*pitch + c] )
//
// One persistent CTA per SM walks a host-built tile list. Warp roles:
//   warp 0      TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx-count)
//   warp 1      MMA issuer    (one thread, tcgen05.mma cta_group::1 kind::f16, M=128 x N=bn x K=16)
//   warps 2..9  epilogue      (tcgen05.ld 32x32b from the double-buffered TMEM accumulator,
//                              bias / time-embedding / border table / gate / GEGLU / residual; the bf16
//                              tile is transposed through swizzled smem so global traffic is coalesced)
// The 3x3 conv is an implicit GEMM: for every tap the A tile is a shifted 4-D TMA box over the NHWC
// activation (out-of-bounds rows/cols are zero-filled by the TMA unit = the conv padding); the
// stride-2 down-sampler conv uses a 5-D view that splits H and W into (index, parity).
// Pruned work is skipped, not multiplied by zero: every expert bucket (segment) has its own kept
// column count, kept K-chunk count and compacted weight block; depth-dropped buckets simply have no
// tiles in the list.
#include "common.cuh"
#include "../../include/aptp_sm100.h"

namespace aptp {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;
constexpr int EPI_PER_QUAD = 3;                    // epilogue warps per TMEM lane quadrant (32-column chunks dealt round-robin)
constexpr int EPI_WARPS = 4 * EPI_PER_QUAD;
constexpr int GEMM_THREADS = 128 + EPI_WARPS * 32;  // warpgroup 0: warp 0 TMA, warp 1 MMA, 2 idle; warps 4..15 epilogue
// registers move from the control warpgroup to the epilogue warpgroups (setmaxnreg): 128 x 56 + 384 x 152 = 64K
#define GEMM_CTRL_REGS "56"
#define GEMM_EPI_REGS "152"
constexpr int TMEM_COLS = 512;
constexpr int STG_WARP_BYTES = 32 * 64;            // per-warp staging: 32 rows x 32 bf16 columns
constexpr int STG_BYTES = EPI_WARPS * STG_WARP_BYTES;
constexpr int MAX_SMEM_SEGS = 96;                   // expert-bucket records cached in shared memory (else read from global)
constexpr int SSEG_BYTES = MAX_SMEM_SEGS * 48;
constexpr int TILE_CACHE = 160;                     // tile records of this CTA staged in shared memory at kernel start
constexpr int STILE_BYTES = TILE_CACHE * 16;
constexpr int SBIAS_BYTES = EPI_WARPS * 128 * 4;    // per epilogue warp: bias slice of its current chunk (32, or 2 x 32 for GEGLU) + the LN-fold column sums

struct GemmParams {
  CUtensorMap tmap_a;
  CUtensorMap tmap_b;
  CUtensorMap tmap_out;  // out_tma: rows x out_ld, box 32 rows x 64 B, 64-byte swizzle (bulk stores of full chunks)
  int out_tma;
  const aptp_gemm_seg* segs;
  const aptp_gemm_tile* tiles;
  int n_tiles;
  int n_segs;
  int a_mode;
  int batch, Ho, Wo;  // OUTPUT spatial size (conv modes)
  int bn, bw, bh, bb;
  int lbw, lbh;       // log2 of the (power-of-two) box extents
  int stages;
  int k_tap_pitch;
  void* out;
  int out_ld, out_mode;
  const float* bias;
  const float* rowvec;
  int rowvec_ld, rows_per_sample;
  const void* residual;  // bf16 rows, or fp32 rows with APTP_EPI_RES_F32 (fp32 residual stream)
  int res_ld;
  const float* gate;
  int gate_ld, gate_group;
  const float* border_tab;
  int tab_ld;
  int flags;
  // LayerNorm folded into this GEMM (APTP_EPI_LN_FOLD): A holds the RAW rows x, the weights are W*gamma, and
  //   out = rstd[row] * (acc - mu[row] * colsum[n]) + bias'[n]
  // with (mu, rstd) derived per row from the (sum, sumsq) partials the PRODUCER of x wrote (rowstat_out below)
  const float* ln_colsum;
  const float2* ln_rowstats;
  // producer side: per-row (sum, sumsq) of every 32-column chunk of the stored values
  float2* rowstat_out;
  int rowstat_chunks;
  // APTP_EPI_GN_STATS: per-channel column sums / sums of squares of every 32-row quadrant of the fp32 output
  float* gn_sum;
  float* gn_sq;
  int gn_ld, gn_blocks;
  // A-stationary mode (linear layers with K <= 6 chunks, i.e. the K = 320 projections of the 64x64 level, which are
  // bound by the L2 -> shared-memory fill, not by the tensor pipe): the host lays the tile list out so that every CTA
  // pair walks all N tiles of one pair of row tiles back to back; the A row tile (128 x K) is loaded ONCE per run
  // (tile flag APTP_TILE_A_FIRST) into a resident region, only the weight tiles stream through the stage ring
  int a_stat;        // 0, or the number of resident A chunk slots
  // Halo mode (2-SM 3x3 stride-1 convs over 8 x 16 pixel boxes): ONE TMA box of 18 rows x 16 pixels x 64 channels per K
  // chunk lands in an A slot and the nine taps are nine MMA groups whose A descriptors start (dy * 16 + dx) pixel rows into
  // it (8-pixel box rows = the 8-row groups of the operand, 16 pixel rows = 2048 B apart); only the weight tiles stream
  // through the ring. A is written to shared memory once per chunk instead of once per tap.
  int halo;          // 0, or the number of A (halo) slots
  // second operand pair of a halo-mode conv (the ResNet's 1x1 shortcut): k2_chunks more K steps per tile whose A tile is
  // the plain 8 x 16-pixel box of a second tensor and whose weights are indexed by the output column
  CUtensorMap tmap_a2;
  CUtensorMap tmap_b2;
  int k2_chunks;
  int* abort_flag;
};

constexpr int A_STAT_MAX_CHUNKS = 6;
constexpr int HALO_W = 16, HALO_H = 18;                   // halo box in pixels (10 needed across; 16 keeps the 8-row groups regular)
constexpr int HALO_BYTES = HALO_W * HALO_H * 128;         // 36 KB per 64-channel chunk (9 boxes of 16 KB before)

// Accumulator columns the MMAs of a tile compute: the LAST column tile of a bucket is ragged (kept widths are not
// multiples of bn), so its MMAs run with N = the 32-column-rounded remainder instead of bn -- tensor time and operand reads
// shrink with it (the weight box is still loaded whole). GEGLU tiles keep bn (their [h | g] halves sit at fixed columns).
// The host may also give a bucket narrower, BALANCED tiles (tile flags bits 8..15 = width / 32: 320 columns under bn = 224
// become 160 + 160 instead of 224 + 96 -- a 96-wide MMA moves the whole A tile for a third of the work).
__device__ __forceinline__ int tile_mma_n(const aptp_gemm_seg& seg, int n0, int bn, bool geglu, int tflags) {
#ifdef APTP_NO_RAGGED_N
  return bn;
#else
  if (geglu) return bn;
  const int w32 = (tflags >> 8) & 0xFF;
  const int width = w32 ? w32 * 32 : bn;
  const int n_cols = seg.n_valid > seg.n_store ? seg.n_valid : seg.n_store;
  const int left = (n_cols - n0 + 31) & ~31;
  return left < width ? (left < 32 ? 32 : left) : width;
#endif
}

__device__ __forceinline__ void advance(int& stage, uint32_t& phase, int stages) {
  if (++stage == stages) {
    stage = 0;
    phase ^= 1;
  }
}

// tile-local row r (0..127) -> global output row; conv tiles are bw x bh x bb pixel boxes.
struct TileGeom {
  int linear;
  int m_base;
  int img0, oy0, ox0;
};
__device__ __forceinline__ int map_row(const GemmParams& p, const TileGeom& g, int r, bool& valid, int& oy,
                                             int& ox) {
  if (g.linear) {
    valid = true;
    oy = ox = 1;
    return g.m_base + r;
  }
  const int ix = r & (p.bw - 1);
  const int iy = (r >> p.lbw) & (p.bh - 1);
  const int ib = r >> (p.lbw + p.lbh);
  oy = g.oy0 + iy;
  ox = g.ox0 + ix;
  const int img = g.img0 + ib;
  valid = (img < p.batch) && (oy < p.Ho) && (ox < p.Wo);
  return (img * p.Ho + oy) * p.Wo + ox;  // output rows < 2^31 (checked on the host)
}

// 32 floats starting at src (all lanes read the same addresses -> L1 broadcast); float4 when aligned.
__device__ __forceinline__ void add32(float* v, const float* __restrict__ src, int n_ok) {
  if (n_ok >= 32 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 f = __ldg(reinterpret_cast<const float4*>(src) + q);
      v[q * 4 + 0] += f.x;
      v[q * 4 + 1] += f.y;
      v[q * 4 + 2] += f.z;
      v[q * 4 + 3] += f.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < n_ok) v[j] += __ldg(src + j);
  }
}

// 32 floats from shared memory (same address in all lanes: broadcast)
__device__ __forceinline__ void add32_smem(float* v, const float* src) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 f = *(reinterpret_cast<const float4*>(src) + q);
    v[q * 4 + 0] += f.x;
    v[q * 4 + 1] += f.y;
    v[q * 4 + 2] += f.z;
    v[q * 4 + 3] += f.w;
  }
}

// folded LayerNorm + bias in two packed FFMA2 per column pair: v = rstd * v + bias' - mu * rstd * colsum
// (bias' and colsum broadcast from shared memory; the epilogue of the K = 320 layers is issue-bound, so the
// fold must cost next to nothing on top of the bias add it replaces)
__device__ __forceinline__ void ln_bias_apply32(float* v, const float* bias, const float* cs, float mu, float rstd) {
  const uint64_t r2 = pack_f32x2(rstd, rstd);
  const float nm = -mu * rstd;
  const uint64_t n2 = pack_f32x2(nm, nm);
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 b = *(reinterpret_cast<const float4*>(bias) + q);
    const float4 c = *(reinterpret_cast<const float4*>(cs) + q);
    uint64_t a0 = fma_f32x2(r2, pack_f32x2(v[q * 4 + 0], v[q * 4 + 1]), pack_f32x2(b.x, b.y));
    uint64_t a1 = fma_f32x2(r2, pack_f32x2(v[q * 4 + 2], v[q * 4 + 3]), pack_f32x2(b.z, b.w));
    a0 = fma_f32x2(n2, pack_f32x2(c.x, c.y), a0);
    a1 = fma_f32x2(n2, pack_f32x2(c.z, c.w), a1);
    unpack_f32x2(a0, v[q * 4 + 0], v[q * 4 + 1]);
    unpack_f32x2(a1, v[q * 4 + 2], v[q * 4 + 3]);
  }
}

// kGeglu selects the GEGLU epilogue (two accumulator halves per output column, erf-GELU) and compiles out the
// residual / row-vector / border-table / fp32 paths it never uses, so neither instantiation pays for the other's
// registers.
//
// kEpi selects the whole output side at compile time -- EPI_BF16 (bf16 rows; bf16 residual, LayerNorm row partials),
// EPI_GEGLU, EPI_F32 (fp32 rows of the residual stream; fp32 residual, GroupNorm column partials), EPI_NCHW (the fp32
// NCHW prediction of conv_out) -- so that no instantiation carries the prefetch registers of another one: with all of
// them in one body the epilogue warps spilled inside the chunk loop (ncu source page, round 2).
enum { EPI_BF16 = 0, EPI_GEGLU = 1, EPI_F32 = 2, EPI_NCHW = 3 };
#ifdef APTP_GEMM_TRACE
// kernel-tuning builds only: cycles each role spends blocked on each barrier, per CTA (tools/gemm_trace.py)
__device__ long long g_gemm_trace[512][16];
#define TRACE_T0() const long long _t0 = clock64(); long long _tw[2] = {0, 0}
#define TRACE_ADD(slot) if (lane == 0) { g_gemm_trace[blockIdx.x][slot] += clock64() - _t0; g_gemm_trace[blockIdx.x][slot + 1] += _tw[1]; if (slot == 2) g_gemm_trace[blockIdx.x][4] += _tw[0]; }
#define TRACE_WAIT(slot, expr) [&]() { const long long _w0 = clock64(); const bool _r = (expr); _tw[slot & 1] += clock64() - _w0; return _r; }()
#else
#define TRACE_T0()
#define TRACE_ADD(slot)
#define TRACE_WAIT(slot, expr) (expr)
#endif
//
// k2Sm: the CTA pair issues ONE tcgen05.mma.cta_group::2 of M = 256 per K step instead of two independent M = 128 MMAs
// over a multicast B tile. Each CTA stages its own A rows and only HALF of the B tile (nothing is duplicated, so the
// ring holds ~1.4x more stages), the leader CTA's full barrier collects the bytes of both CTAs, the leader issues the
// MMAs and multicasts the commits, and the epilogue warps of both CTAs release the accumulator on the leader's
// barrier. Per MMA an SM reads A + B/2 instead of A + B from shared memory -- the operand fetch of a 128 x 160 tile
// alone took 115 of the 128 B/clk of shared-memory bandwidth and left nothing for the TMA writes and the epilogue's
// staging (round-2 analysis, DESIGN.md section 5).
template <int kEpi, bool k2Sm>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
grouped_gemm_kernel(const __grid_constant__ GemmParams p) {
  constexpr bool kGeglu = (kEpi == EPI_GEGLU);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stages = p.stages;
  // normal mode: ring of (A tile | B tile) stages; A-stationary: a_stat resident A chunk slots, then a ring of B tiles
  const uint32_t stage_bytes = ((p.a_stat || p.halo) ? 0u : (uint32_t)A_STAGE_BYTES) + (uint32_t)p.bn * (k2Sm ? 64u : 128u);
  const uint32_t ring_off = p.halo ? (uint32_t)p.halo * HALO_BYTES : (uint32_t)p.a_stat * A_STAGE_BYTES;
  uint8_t* stg_base = smem + ring_off + (size_t)stages * stage_bytes;
  float* sbias = reinterpret_cast<float*>(stg_base + STG_BYTES);
  aptp_gemm_seg* ssegs = reinterpret_cast<aptp_gemm_seg*>(stg_base + STG_BYTES + SBIAS_BYTES);
  aptp_gemm_tile* stiles = reinterpret_cast<aptp_gemm_tile*>(stg_base + STG_BYTES + SBIAS_BYTES + SSEG_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stg_base + STG_BYTES + SBIAS_BYTES + SSEG_BYTES + STILE_BYTES);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* tfull_bar = empty_bar + stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* afull_bar = tempty_bar + 2;                   // A-stationary: one pair of barriers per resident A chunk
  uint64_t* aempty_bar = afull_bar + A_STAT_MAX_CHUNKS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty_bar + A_STAT_MAX_CHUNKS);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
#ifdef APTP_GEMM_TRACE
  const long long _t0_epi = clock64();
#endif
  // CTA pair (cluster of 2): the pair works on tiles (2i, 2i+1) of the list, which share the expert bucket and
  // the weight rows (n0) and differ in their 128 output rows; each CTA fetches HALF of the weight tile of every
  // stage and multicasts it to both, so the L2 -> shared-memory traffic for B is halved.
  // (rank / pair bookkeeping is recomputed inside each role: values kept live across the setmaxnreg split are
  // spilled to local memory by ptxas and reloaded in the hot loops)
#define GEMM_ROLE_PROLOGUE()                                                                        \
  const uint32_t cta_rank = cluster_ctarank();                                                      \
  const int pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1, n_pairs = p.n_tiles >> 1;        \
  const aptp_gemm_seg* segs = (p.n_segs <= MAX_SMEM_SEGS) ? ssegs : p.segs;                         \
  const uint32_t tmem_base = *tmem_slot;                                                            \
  (void)cta_rank; (void)pair0; (void)pair_stride; (void)n_pairs; (void)segs; (void)tmem_base;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_a);
    tma_prefetch_desc(&p.tmap_b);
    if (p.out_tma) tma_prefetch_desc(&p.tmap_out);
    if (p.k2_chunks) {
      tma_prefetch_desc(&p.tmap_a2);
      tma_prefetch_desc(&p.tmap_b2);
    }
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < stages; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], k2Sm ? 1 : 2);  // one tcgen05.commit from each CTA of the pair (2-SM: the leader's)
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(&tfull_bar[a], 1);
        mbar_init(&tempty_bar[a], k2Sm ? 2 * EPI_WARPS : EPI_WARPS);  // 2-SM: both CTAs' warps, on the leader
      }
      for (int a = 0; a < A_STAT_MAX_CHUNKS; ++a) {
        mbar_init(&afull_bar[a], 1);
        mbar_init(&aempty_bar[a], 1);
      }
      fence_barrier_init();
    }
    __syncwarp();
    if constexpr (k2Sm) {
      tmem_alloc_2sm(tmem_slot, TMEM_COLS);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(tmem_slot, TMEM_COLS);
      tmem_relinquish();
    }
  }
  // expert-bucket records -> shared memory (every role reads one per tile; a dependent global load per tile
  // is a ~1 us bubble on the short K=320 tiles)
  const bool segs_in_smem = p.n_segs <= MAX_SMEM_SEGS;
  if (segs_in_smem) {
    const int4* src = reinterpret_cast<const int4*>(p.segs);
    int4* dst = reinterpret_cast<int4*>(ssegs);
    for (int i = threadIdx.x; i < p.n_segs * 3; i += blockDim.x) dst[i] = __ldg(src + i);
  }
  // ... and so are this CTA's first TILE_CACHE tile records: each role used to prefetch its next record into
  // registers, but in the register-starved epilogue warps ptxas spilled that prefetch to local memory, which turns it
  // into a blocking ~1 us load per tile (ncu source page, round 2). Records beyond the cache are read from global.
  {
    const int pair0_ = blockIdx.x >> 1, pair_stride_ = gridDim.x >> 1, n_pairs_ = p.n_tiles >> 1;
    const uint32_t rank_ = cluster_ctarank();
    const int4* src = reinterpret_cast<const int4*>(p.tiles);
    int4* dst = reinterpret_cast<int4*>(stiles);
    for (int i = threadIdx.x; i < TILE_CACHE; i += blockDim.x) {
      const int pr = pair0_ + i * pair_stride_;
      if (pr < n_pairs_) dst[i] = __ldg(src + 2 * pr + rank_);
    }
  }
  tc_fence_before();
  cluster_sync_all();  // barriers of BOTH CTAs are initialised before any multicast load / remote arrive
  tc_fence_after();
  pdl_launch();  // the next kernel's CTAs may take over SMs as ours exit and run their prologue
  pdl_wait();    // everything above touched only launch-time data; from here on we read what predecessors wrote

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 " GEMM_CTRL_REGS ";");
  if (warp == 0) {
    // ------------------------------- TMA producer -------------------------------
    // Whole warp in uniform control flow, one elected lane issues (see the MMA issuer for why).
    {
      GEMM_ROLE_PROLOGUE();
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      const int taps = (p.a_mode == APTP_A_LINEAR) ? 1 : 9;
      const uint32_t b_half_bytes = (uint32_t)p.bn * 64u;          // bn/2 weight rows x 128 B
      uint32_t a_bits = 0;  // A-stationary: bit kc = parity of the uses of resident chunk kc (runs may differ in K)
      int aslot = 0;        // halo mode: A slot ring
      uint32_t aphase = 0;
      int ti = 0;
      TRACE_T0();
      for (int pr = pair0; pr < n_pairs && ok; pr += pair_stride, ++ti) {
        const aptp_gemm_tile tile = (ti < TILE_CACHE) ? stiles[ti] : p.tiles[2 * pr + cta_rank];
        if (tile.flags & APTP_TILE_SKIP) continue;
        const aptp_gemm_seg seg = segs[tile.seg];
        if (!k2Sm && p.a_stat) {
          const int b_row = seg.w_row_off + tile.n0 + (int)cta_rank * (p.bn >> 1);
          if (tile.flags & APTP_TILE_A_FIRST) {
            // the A row tile of this run: chunk kc may be overwritten as soon as the previous run's last N tile has
            // consumed it (per-chunk barriers, so the refill trails the tensor pipe chunk by chunk)
            for (int kc = 0; kc < seg.k_chunks && ok; ++kc) {
              if (!mbar_wait(&aempty_bar[kc], ((a_bits >> kc) & 1u) ^ 1u, p.abort_flag)) {
                ok = false;
                break;
              }
              a_bits ^= 1u << kc;
              if (elect_one()) {
                mbar_expect_tx(&afull_bar[kc], A_STAGE_BYTES);
                tma_load_2d(smem + (size_t)kc * A_STAGE_BYTES, &p.tmap_a, &afull_bar[kc], kc * BK, tile.m_base);
              }
              __syncwarp();
            }
          }
          for (int kc = 0; kc < seg.k_chunks && ok; ++kc) {
            if (!mbar_wait(&empty_bar[stage], phase ^ 1, p.abort_flag)) {
              ok = false;
              break;
            }
            if (elect_one()) {
              uint8_t* sb = smem + ring_off + (size_t)stage * stage_bytes;
              mbar_expect_tx(&full_bar[stage], stage_bytes);
              tma_load_2d_mc(sb + cta_rank * b_half_bytes, &p.tmap_b, &full_bar[stage], kc * BK, b_row, (uint16_t)0x3);
            }
            __syncwarp();
            advance(stage, phase, stages);
          }
          continue;
        }
        int img = 0, oy0 = 0, ox0 = 0;
        if (p.a_mode != APTP_A_LINEAR) {
          const int hw = p.Ho * p.Wo;
          img = tile.m_base / hw;
          const int rem = tile.m_base - img * hw;
          oy0 = rem / p.Wo;
          ox0 = rem - oy0 * p.Wo;
        }
        // this CTA's half of the weight tile (2-SM: half of the columns the tile's MMAs really compute)
        const int b_row = seg.w_row_off + tile.n0 +
                          (int)cta_rank * ((k2Sm ? tile_mma_n(seg, tile.n0, p.bn, kGeglu, tile.flags) : p.bn) >> 1);
        if constexpr (k2Sm) {
          if (p.halo) {
            for (int kc = 0; kc < seg.k_chunks && ok; ++kc) {
              if (!mbar_wait(&aempty_bar[aslot], aphase ^ 1, p.abort_flag)) {
                ok = false;
                break;
              }
              if (elect_one()) {
                if (cta_rank == 0) mbar_expect_tx(&afull_bar[aslot], 2u * HALO_BYTES);
                tma_load_4d_2sm(smem + (size_t)aslot * HALO_BYTES, &p.tmap_a, &afull_bar[aslot], kc * BK, ox0 - 1, oy0 - 1, img);
              }
              __syncwarp();
              for (int tap = 0; tap < 9; ++tap) {
                if (!mbar_wait(&empty_bar[stage], phase ^ 1, p.abort_flag)) {
                  ok = false;
                  break;
                }
                if (elect_one()) {
                  if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2u * stage_bytes);
                  tma_load_2d_2sm(smem + ring_off + (size_t)stage * stage_bytes, &p.tmap_b, &full_bar[stage],
                                  tap * p.k_tap_pitch + kc * BK, b_row);
                }
                __syncwarp();
                advance(stage, phase, stages);
              }
              if (++aslot == p.halo) {
                aslot = 0;
                aphase ^= 1;
              }
            }
            // the 1x1 shortcut's K steps: plain box of the second tensor into the next A slot, W2 rows = output columns
            // of this bucket's block in w2 (per-expert shortcut weights). GEGLU launches never carry a2 (the launcher
            // refuses it); not reading the offset there keeps that instantiation at the parent's 0 spill bytes.
            const int b2_row = (kGeglu ? 0 : seg.w2_row_off) + tile.n0 +
                               (int)cta_rank * (tile_mma_n(seg, tile.n0, p.bn, kGeglu, tile.flags) >> 1);
            for (int kc = 0; kc < p.k2_chunks && ok; ++kc) {
              if (!mbar_wait(&aempty_bar[aslot], aphase ^ 1, p.abort_flag) ||
                  !mbar_wait(&empty_bar[stage], phase ^ 1, p.abort_flag)) {
                ok = false;
                break;
              }
              if (elect_one()) {
                if (cta_rank == 0) {
                  mbar_expect_tx(&afull_bar[aslot], 2u * A_STAGE_BYTES);
                  mbar_expect_tx(&full_bar[stage], 2u * stage_bytes);
                }
                tma_load_4d_2sm(smem + (size_t)aslot * HALO_BYTES, &p.tmap_a2, &afull_bar[aslot], kc * BK, ox0, oy0, img);
                tma_load_2d_2sm(smem + ring_off + (size_t)stage * stage_bytes, &p.tmap_b2, &full_bar[stage], kc * BK, b2_row);
              }
              __syncwarp();
              advance(stage, phase, stages);
              if (++aslot == p.halo) {
                aslot = 0;
                aphase ^= 1;
              }
            }
            continue;
          }
        }
        for (int tap = 0; tap < taps && ok; ++tap) {
          const int dy = tap / 3, dx = tap - dy * 3;
          for (int kc = 0; kc < seg.k_chunks; ++kc) {
            if (!TRACE_WAIT(1, mbar_wait(&empty_bar[stage], phase ^ 1, p.abort_flag))) {
              ok = false;
              break;
            }
            if (elect_one()) {
              uint8_t* sa = smem + (size_t)stage * stage_bytes;
              uint8_t* sb = sa + A_STAGE_BYTES;
              // input y = 2*oy + dy - 1: dy=0 -> (parity 1, shift -1); dy=1 -> (0, 0); dy=2 -> (1, 0)
              const int py = (dy == 1) ? 0 : 1, sy = (dy == 0) ? -1 : 0;
              const int px = (dx == 1) ? 0 : 1, sx = (dx == 0) ? -1 : 0;
              if constexpr (k2Sm) {
                // the LEADER's barrier counts the bytes both CTAs deliver for this stage (its own expect_tx may come
                // after the peer's bytes: the transaction count is signed and the phase cannot complete before the
                // leader's arrival)
                if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2u * stage_bytes);
                if (p.a_mode == APTP_A_LINEAR) {
                  tma_load_2d_2sm(sa, &p.tmap_a, &full_bar[stage], kc * BK, tile.m_base);
                } else if (p.a_mode == APTP_A_CONV3X3) {
                  tma_load_4d_2sm(sa, &p.tmap_a, &full_bar[stage], kc * BK, ox0 + dx - 1, oy0 + dy - 1, img);
                } else {
                  tma_load_5d_2sm(sa, &p.tmap_a, &full_bar[stage], px * p.k_tap_pitch + kc * BK, ox0 + sx, py, oy0 + sy,
                                  img);
                }
                tma_load_2d_2sm(sb, &p.tmap_b, &full_bar[stage], tap * p.k_tap_pitch + kc * BK, b_row);
              } else {
                mbar_expect_tx(&full_bar[stage], stage_bytes);
                if (p.a_mode == APTP_A_LINEAR) {
                  tma_load_2d(sa, &p.tmap_a, &full_bar[stage], kc * BK, tile.m_base);
                } else if (p.a_mode == APTP_A_CONV3X3) {
                  tma_load_4d(sa, &p.tmap_a, &full_bar[stage], kc * BK, ox0 + dx - 1, oy0 + dy - 1, img);
                } else {
                  tma_load_5d(sa, &p.tmap_a, &full_bar[stage], px * p.k_tap_pitch + kc * BK, ox0 + sx, py, oy0 + sy,
                              img);
                }
                tma_load_2d_mc(sb + cta_rank * b_half_bytes, &p.tmap_b, &full_bar[stage],
                               tap * p.k_tap_pitch + kc * BK, b_row, (uint16_t)0x3);
              }
            }
            __syncwarp();
            advance(stage, phase, stages);
          }
        }
      }
      TRACE_ADD(0);
    }
  } else if (warp == 1 && (!k2Sm || cluster_ctarank() == 0)) {
    // ------------------------------- MMA issuer ---------------------------------
    // (2-SM: the leader CTA issues for the pair; the peer's warp 1 only allocates and frees tensor memory)
    // The WHOLE warp walks the tile list in uniform control flow (so descriptors, barrier addresses and
    // loop counters live in uniform registers) and one elected lane issues the tcgen05 instructions.
    // A loop nested under `if (lane == 0)` instead makes ptxas wrap every UTCHMMA in a per-lane
    // R2UR "waterfall" loop, which capped the issue rate at ~140 cycles per MMA (ncu, round 1).
    {
      GEMM_ROLE_PROLOGUE();
      const uint32_t smem_base = smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      bool ok = true;
      uint32_t a_bits = 0;
      int aslot = 0;
      uint32_t aphase = 0;
      int ti = 0;
      TRACE_T0();
      for (int pr = pair0; pr < n_pairs && ok; pr += pair_stride, ++ti) {
        const aptp_gemm_tile* trec = (ti < TILE_CACHE) ? &stiles[ti] : &p.tiles[2 * pr + cta_rank];
        const int seg_id = __shfl_sync(0xffffffffu, trec->seg, 0);
        const int tflags = __shfl_sync(0xffffffffu, trec->flags, 0);
        if (tflags & APTP_TILE_SKIP) continue;
        const int k_chunks = __shfl_sync(0xffffffffu, segs[seg_id].k_chunks, 0);
        const int n_mma = __shfl_sync(0xffffffffu, tile_mma_n(segs[seg_id], trec->n0, p.bn, kGeglu, tflags), 0);
        const uint32_t idesc = make_idesc_bf16(k2Sm ? 2 * BM : BM, (uint32_t)n_mma, 0, 0);
        const int kblocks = ((p.a_mode == APTP_A_LINEAR) ? 1 : 9) * k_chunks;
        if (!TRACE_WAIT(3, mbar_wait(&tempty_bar[acc], acc_phase ^ 1, p.abort_flag))) break;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.bn);
        if (!k2Sm && p.a_stat) {
          const bool first = (tflags & APTP_TILE_A_FIRST) != 0, last = (tflags & APTP_TILE_A_LAST) != 0;
          for (int kc = 0; kc < k_chunks; ++kc) {
            if (first) {
              if (!mbar_wait(&afull_bar[kc], (a_bits >> kc) & 1u, p.abort_flag)) {
                ok = false;
                break;
              }
              a_bits ^= 1u << kc;
            }
            if (!mbar_wait(&full_bar[stage], phase, p.abort_flag)) {
              ok = false;
              break;
            }
            tc_fence_after();
            const uint64_t da = make_desc_kmajor_sw128(smem_base + (uint32_t)kc * A_STAGE_BYTES);
            const uint64_t db = make_desc_kmajor_sw128(smem_base + ring_off + (uint32_t)stage * stage_bytes);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k)
                umma_bf16_ss(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kc | k) != 0 ? 1u : 0u);
              umma_commit_mc(&empty_bar[stage], (uint16_t)0x3);
              if (last) umma_commit(&aempty_bar[kc]);  // the run's last N tile: chunk kc may be refilled
            }
            __syncwarp();
            advance(stage, phase, stages);
          }
          if (!ok) break;
          if (elect_one()) umma_commit(&tfull_bar[acc]);
          __syncwarp();
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
          continue;
        }
        if constexpr (k2Sm) {
          if (p.halo) {
            for (int kc = 0; kc < k_chunks && ok; ++kc) {
              if (!mbar_wait(&afull_bar[aslot], aphase, p.abort_flag)) {
                ok = false;
                break;
              }
              for (int tap = 0; tap < 9; ++tap) {
                if (!TRACE_WAIT(4, mbar_wait(&full_bar[stage], phase, p.abort_flag))) {
                  ok = false;
                  break;
                }
                tc_fence_after();
                const int dy = tap / 3, dx = tap - dy * 3;
                // output pixel (y, x) of the 8 x 16 box reads halo pixel (y + dy, x + dx): rows of 16 pixels = 2048 B
                const uint64_t da = make_desc_kmajor_sw128_ex(
                    smem_base + (uint32_t)aslot * HALO_BYTES + (uint32_t)(dy * HALO_W + dx) * 128u, HALO_W * 128u);
                const uint64_t db = make_desc_kmajor_sw128(smem_base + ring_off + (uint32_t)stage * stage_bytes);
                if (elect_one()) {
#pragma unroll
                  for (int k = 0; k < BK / 16; ++k)
                    umma_bf16_ss_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kc | tap | k) != 0 ? 1u : 0u);
                  umma_commit_2sm(&empty_bar[stage], (uint16_t)0x3);
                }
                __syncwarp();
                advance(stage, phase, stages);
              }
              if (!ok) break;
              if (elect_one()) umma_commit_2sm(&aempty_bar[aslot], (uint16_t)0x3);  // both CTAs' halo slot may be refilled
              __syncwarp();
              if (++aslot == p.halo) {
                aslot = 0;
                aphase ^= 1;
              }
            }
            for (int kc = 0; kc < p.k2_chunks && ok; ++kc) {  // the 1x1 shortcut accumulates into the same tile
              if (!mbar_wait(&afull_bar[aslot], aphase, p.abort_flag) ||
                  !TRACE_WAIT(4, mbar_wait(&full_bar[stage], phase, p.abort_flag))) {
                ok = false;
                break;
              }
              tc_fence_after();
              const uint64_t da = make_desc_kmajor_sw128(smem_base + (uint32_t)aslot * HALO_BYTES);
              const uint64_t db = make_desc_kmajor_sw128(smem_base + ring_off + (uint32_t)stage * stage_bytes);
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < BK / 16; ++k)
                  umma_bf16_ss_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, 1u);
                umma_commit_2sm(&empty_bar[stage], (uint16_t)0x3);
                umma_commit_2sm(&aempty_bar[aslot], (uint16_t)0x3);
              }
              __syncwarp();
              advance(stage, phase, stages);
              if (++aslot == p.halo) {
                aslot = 0;
                aphase ^= 1;
              }
            }
            if (!ok) break;
            if (elect_one()) umma_commit_2sm(&tfull_bar[acc], (uint16_t)0x3);
            __syncwarp();
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
            continue;
          }
        }
        for (int kb = 0; kb < kblocks; ++kb) {
          if (!TRACE_WAIT(4, mbar_wait(&full_bar[stage], phase, p.abort_flag))) {
            ok = false;
            break;
          }
          tc_fence_after();
          const uint32_t a_addr = smem_base + (uint32_t)stage * stage_bytes;
          const uint64_t da = make_desc_kmajor_sw128(a_addr);
          const uint64_t db = make_desc_kmajor_sw128(a_addr + A_STAGE_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // +32 bytes per K=16 step inside the 128B-swizzled row: +2 in the (addr >> 4) field
              if constexpr (k2Sm)
                umma_bf16_ss_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
              else
                umma_bf16_ss(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
            }
            // the stage is free once BOTH CTAs have read it (2-SM: one commit covers the pair's MMAs)
            if constexpr (k2Sm) umma_commit_2sm(&empty_bar[stage], (uint16_t)0x3);
            else umma_commit_mc(&empty_bar[stage], (uint16_t)0x3);
          }
          __syncwarp();
          advance(stage, phase, stages);
        }
        if (!ok) break;
        if (elect_one()) {
          if constexpr (k2Sm) umma_commit_2sm(&tfull_bar[acc], (uint16_t)0x3);  // both CTAs' epilogues
          else umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
      TRACE_ADD(2);
    }
  }
  } else {
    // ------------------------------- epilogue -----------------------------------
    asm volatile("setmaxnreg.inc.sync.aligned.u32 " GEMM_EPI_REGS ";");
    GEMM_ROLE_PROLOGUE();
    // Thread = one accumulator row (TMEM lane). Results are transposed through a per-warp swizzled
    // smem tile so that every global store / residual load instruction covers 8 rows x 64 contiguous
    // bytes (full sectors) instead of 32 rows x 16 bytes.
    const int ew = warp - 4;
    const int quad = warp & 3;       // TMEM lane quadrant this warp may touch
    const int cpar = ew >> 2;        // position of this warp among the EPI_PER_QUAD warps of its quadrant
    float* wbias = sbias + ew * 128;
    uint32_t chunk_rot = 0;          // chunks dealt so far (mod EPI_PER_QUAD): keeps the deal balanced across tiles
    const int r_own = quad * 32 + lane;
    uint8_t* stg = stg_base + ew * STG_WARP_BYTES;
    // staging addresses: own row (write side) and the coalesced (8 rows x 4 x 16 B) side
    const uint32_t stg_own = smem_u32(stg) + lane * 64;
    const int own_sw = (lane >> 1) & 3;
    const int co_q = lane & 3;  // 16-byte column unit handled by this lane on the coalesced side
    int acc = 0;
    uint32_t acc_phase = 0;
    constexpr bool geglu = kGeglu;
    constexpr bool bf16_out = (kEpi == EPI_BF16 || kEpi == EPI_GEGLU);
    int ti = 0;
    bool st_pending = false;
#ifdef APTP_GEMM_TRACE
    long long _tr_ld = 0, _tr_math = 0, _tr_st = 0, _tr_tfull = 0, _tr_busy = 0, _tr_tiles = 0;
#endif
    for (int pr = pair0; pr < n_pairs; pr += pair_stride, ++ti) {
      const aptp_gemm_tile tile = (ti < TILE_CACHE) ? stiles[ti] : p.tiles[2 * pr + cta_rank];
      if (tile.flags & APTP_TILE_SKIP) continue;  // padding entry of an A-stationary tile list
      const aptp_gemm_seg seg = segs[tile.seg];
      const bool placeholder = (tile.flags & APTP_TILE_PLACEHOLDER) != 0;  // odd tile count of a bucket: no stores
      TileGeom g;
      g.linear = (p.a_mode == APTP_A_LINEAR);
      g.m_base = tile.m_base;
      g.img0 = g.oy0 = g.ox0 = 0;
      if (!g.linear) {
        const int hw = p.Ho * p.Wo;
        g.img0 = tile.m_base / hw;
        const int rem = tile.m_base - g.img0 * hw;
        g.oy0 = rem / p.Wo;
        g.ox0 = rem - g.oy0 * p.Wo;
      }
      // ---- own row ----
      bool valid;
      int oy, ox;
      const int row = map_row(p, g, r_own, valid, oy, ox);
      valid = valid && !placeholder && (row < seg.row_end) && (row >= seg.row_begin);
      const int sample = valid ? row / p.rows_per_sample : 0;
      const int ycls = g.linear ? 1 : ((oy == 0) ? 0 : ((oy == p.Ho - 1) ? 2 : 1));
      const int xcls = g.linear ? 1 : ((ox == 0) ? 0 : ((ox == p.Wo - 1) ? 2 : 1));
      const float* tabp =
          (!kGeglu && p.border_tab) ? p.border_tab + seg.tab_off + (size_t)(ycls * 3 + xcls) * p.tab_ld : nullptr;
      // ---- the 4 rows this lane moves on the coalesced side ----
      int co_row[4];
      bool co_ok[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        int a, b;
        bool v;
        const int rr = map_row(p, g, quad * 32 + it * 8 + (lane >> 2), v, a, b);
        co_ok[it] = v && !placeholder && (rr < seg.row_end) && (rr >= seg.row_begin);
        co_row[it] = rr;
      }
      const int ocol_base = geglu ? tile.n0 / 2 : tile.n0;  // first OUTPUT column of this tile
      // bulk (TMA) store of a chunk: all 32 rows of this quadrant lie inside the bucket (linear layers; ragged bucket
      // ends, placeholders and partial column chunks take the per-lane store path)
      const int row0_q = tile.m_base + quad * 32;
      const bool rows_full = bf16_out && p.out_tma && !placeholder && row0_q >= seg.row_begin && row0_q + 32 <= seg.row_end;
      // GroupNorm partial statistics: row of the partial planes this (tile, quadrant) owns
      long long gn_row = -1;
      if ((kEpi == EPI_F32 || kEpi == EPI_BF16) && p.gn_sum != nullptr && !placeholder) {
        const int smp = tile.m_base / p.rows_per_sample;
        const int rem = tile.m_base - smp * p.rows_per_sample;
        int t_in_s;
        if (g.linear) {
          t_in_s = rem >> 7;
        } else {
          const int oy0 = rem / p.Wo, ox0 = rem - oy0 * p.Wo;
          t_in_s = (oy0 >> p.lbh) * (p.Wo >> p.lbw) + (ox0 >> p.lbw);
        }
        gn_row = ((long long)smp * p.gn_blocks + t_in_s * 4 + quad) * p.gn_ld;
      }

      // residual of the first chunk goes in flight before we wait for the accumulator
      uint4 rres[kEpi == EPI_BF16 ? 4 : 1];
      const bool use_res = (kEpi == EPI_BF16) && (p.residual != nullptr);
      auto load_res = [&](int col0) {
        if constexpr (kEpi == EPI_BF16) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            rres[it] = make_uint4(0u, 0u, 0u, 0u);
            if (co_ok[it] && col0 + co_q * 8 < seg.n_valid)
              rres[it] = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.residual) +
                                                         (size_t)co_row[it] * p.res_ld + seg.out_col_off + col0 +
                                                         co_q * 8);  // may alias `out`
          }
        }
      };
      // fp32 residual stream (block outputs, DESIGN.md section 4): same coalesced shape as the bf16 path -- one
      // instruction moves 8 rows x 64 contiguous bytes -- but 64 B are 16 fp32 columns, so a 32-column chunk goes
      // through the per-warp staging tile as two halves. The chunk's residual is loaded one chunk ahead.
      constexpr bool f32_rows = (kEpi == EPI_F32);
      const bool use_res32 = f32_rows && (p.residual != nullptr) && (p.flags & APTP_EPI_RES_F32) != 0;
      uint4 rres32[f32_rows ? 2 : 1][f32_rows ? 4 : 1];
      auto load_res32 = [&](int col0) {
        if constexpr (f32_rows) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              rres32[h][it] = make_uint4(0u, 0u, 0u, 0u);
              if (co_ok[it] && col0 + h * 16 + co_q * 4 < seg.n_valid)
                rres32[h][it] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.residual) +
                                                                (size_t)co_row[it] * p.res_ld + seg.out_col_off + col0 +
                                                                h * 16 + co_q * 4);  // may alias `out`
            }
        }
      };
      // this tile's chunks are dealt round-robin to the EPI_PER_QUAD warps of the quadrant, continuing where the
      // previous tile stopped, so tiles whose chunk count is not a multiple of EPI_PER_QUAD still balance
      const int w32_tile = (tile.flags >> 8) & 0xFF;  // balanced tiles: narrower than bn
      const int out_cols_per_tile = geglu ? p.bn / 2 : (w32_tile ? w32_tile * 32 : p.bn);
      const int n_chunks = (out_cols_per_tile + 31) >> 5;
      const int c_first = (cpar + EPI_PER_QUAD - (int)(chunk_rot % EPI_PER_QUAD)) % EPI_PER_QUAD;
      chunk_rot += (uint32_t)n_chunks;
      // bias slice of a chunk: one coalesced load per lane, issued early; broadcast through smem at use
      const bool ln_fold = (p.flags & APTP_EPI_LN_FOLD) != 0;
      float bias_h = 0.f, bias_g = 0.f, cs_h = 0.f, cs_g = 0.f;
      auto load_bias = [&](int c) {
        const int col0 = ocol_base + c * 32;
        bias_h = bias_g = cs_h = cs_g = 0.f;
        if (p.bias && col0 + lane < seg.n_valid) {
          if (geglu) {  // packed bias follows the packed (interleaved [h | g]) weight rows
            bias_h = __ldg(p.bias + seg.vec_off + tile.n0 + c * 32 + lane);
            bias_g = __ldg(p.bias + seg.vec_off + tile.n0 + p.bn / 2 + c * 32 + lane);
          } else {
            bias_h = __ldg(p.bias + seg.vec_off + col0 + lane);
          }
        }
        if (ln_fold && col0 + lane < seg.n_valid) {
          if (geglu) {
            cs_h = __ldg(p.ln_colsum + seg.vec_off + tile.n0 + c * 32 + lane);
            cs_g = __ldg(p.ln_colsum + seg.vec_off + tile.n0 + p.bn / 2 + c * 32 + lane);
          } else {
            cs_h = __ldg(p.ln_colsum + seg.vec_off + col0 + lane);
          }
        }
      };
      // folded LayerNorm: this row's (mean, rstd), one 8-byte load per tile, in flight under the accumulator wait
      float ln_mu = 0.f, ln_rstd = 1.f;
      if (ln_fold && valid) {
        const float2 ms = __ldg(p.ln_rowstats + row);
        ln_mu = ms.x;
        ln_rstd = ms.y;
      }
      if (c_first < n_chunks) {
        if (use_res && ocol_base + c_first * 32 < seg.n_store) load_res(ocol_base + c_first * 32);
        if (use_res32 && ocol_base + c_first * 32 < seg.n_store) load_res32(ocol_base + c_first * 32);
        load_bias(c_first);
      }

#ifdef APTP_GEMM_TRACE
      const long long _e0 = clock64();
      const bool got = mbar_wait(&tfull_bar[acc], acc_phase, p.abort_flag);
      const long long _e1 = clock64();
      _tr_tfull += _e1 - _e0;
#else
      const bool got = mbar_wait(&tfull_bar[acc], acc_phase, p.abort_flag);
#endif
      if (!got) break;
      tc_fence_after();
      // first use of the prefetched row statistics stays BEHIND the wait (ptxas otherwise hoists -mu * rstd above it and
      // the warp blocks on the load before it ever looks at the barrier)
      asm volatile("" : "+f"(ln_mu), "+f"(ln_rstd));
      // this warp's arrive on tempty_bar[acc]. Releasing right after the warp's LAST TMEM read of the tile
      // (-DAPTP_EARLY_RELEASE) instead of after its stores was measured SLOWER on the K = 320 layers (the MMA running
      // further ahead only adds operand traffic to a shared-memory pipe the epilogue staging also needs), so the
      // release stays at the end of the tile.
      bool released = false;
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (k2Sm) mbar_arrive_rank(&tempty_bar[acc], 0u);  // the leader's MMA warp waits for both CTAs
          else mbar_arrive(&tempty_bar[acc]);
        }
      };
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * p.bn);

#ifdef APTP_DBG_NOEPI  // kernel-tuning build (tools/build_variant.sh): main loop alone, no epilogue work at all (DESIGN 9a)
      if (p.n_tiles < 0)
#endif
      for (int c = c_first; c < n_chunks; c += EPI_PER_QUAD) {
        const int col0 = ocol_base + c * 32;
        if (col0 >= seg.n_store) break;  // warp-uniform
        const int n_ok = seg.n_valid - col0;  // columns of this chunk that carry data (may be <= 0)
        if (st_pending) {  // the previous chunk's bulk store must have read the staging tile before it is rewritten
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
          st_pending = false;
        }
        if (p.bias || ln_fold) {
          wbias[lane] = bias_h;
          if (geglu) wbias[32 + lane] = bias_g;
          if (ln_fold) {
            wbias[64 + lane] = cs_h;
            if (geglu) wbias[96 + lane] = cs_g;
          }
          __syncwarp();
        }
        const bool more = (c + EPI_PER_QUAD < n_chunks) && (col0 + 32 * EPI_PER_QUAD < seg.n_store);
        float v[32];
#ifdef APTP_GEMM_TRACE
        const long long _c0 = clock64();
        long long _c1 = 0;
#define TRACE_LD_DONE() _c1 = clock64(); _tr_ld += _c1 - _c0
#else
#define TRACE_LD_DONE()
#endif
        if constexpr (kGeglu) {
          uint32_t ra[32], rb[32];
          tmem_ld_32x32(t_addr + c * 32, ra);
          tmem_ld_32x32(t_addr + p.bn / 2 + c * 32, rb);
          tmem_ld_wait();
          TRACE_LD_DONE();
#ifdef APTP_EARLY_RELEASE
          if (!more) {
            release_acc();
            released = true;
          }
#endif
          float gv[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            v[j] = __uint_as_float(ra[j]);
            gv[j] = __uint_as_float(rb[j]);
          }
          if (ln_fold) {  // (host: APTP_EPI_LN_FOLD always comes with a bias vector)
            ln_bias_apply32(v, wbias, wbias + 64, ln_mu, ln_rstd);
            ln_bias_apply32(gv, wbias + 32, wbias + 96, ln_mu, ln_rstd);
          } else if (p.bias) {
            add32_smem(v, wbias);
            add32_smem(gv, wbias + 32);
          }
          if (p.gate && valid) {
            const float* gp = p.gate + (size_t)sample * p.gate_ld;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (j < n_ok) {
                const float gs = __ldg(gp + (col0 + j) / p.gate_group);
                v[j] *= gs;
                gv[j] *= gs;
              }
            }
          }
#ifdef APTP_GEGLU_AS
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] *= gelu_erf_fast(gv[j]);
#else
#pragma unroll
          for (int j = 0; j < 32; j += 2) geglu_pair(v[j], v[j + 1], gv[j], gv[j + 1]);
#endif
          if (p.bias || ln_fold) {
            __syncwarp();
            if (more) load_bias(c + EPI_PER_QUAD);
          }
        } else {
          uint32_t ra[32];
          tmem_ld_32x32(t_addr + c * 32, ra);
          tmem_ld_wait();
          TRACE_LD_DONE();
#ifdef APTP_EARLY_RELEASE
          if (!more) {
            release_acc();
            released = true;
          }
#endif
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(ra[j]);
          if (ln_fold) ln_bias_apply32(v, wbias, wbias + 64, ln_mu, ln_rstd);
          else if (p.bias) add32_smem(v, wbias);
          if (p.bias || ln_fold) {
            __syncwarp();
            if (more) load_bias(c + EPI_PER_QUAD);
          }
          if (p.rowvec && valid) add32(v, p.rowvec + (size_t)sample * p.rowvec_ld + col0, n_ok);
          if (tabp) add32(v, tabp + col0, n_ok);
          if (p.gate && valid) {
            const float* gp = p.gate + (size_t)sample * p.gate_ld;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < n_ok) v[j] *= __ldg(gp + (col0 + j) / p.gate_group);
          }
          if (p.flags & APTP_EPI_SILU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = silu_f(v[j]);
          }
        }

#ifdef APTP_GEMM_TRACE
        const long long _c2 = clock64();
        _tr_math += _c2 - _c1;
#endif
        if constexpr (bf16_out) {
          // per-warp staging tile: 32 rows x 64 B, 16-byte units XOR-swizzled by (row >> 1) & 3. Plain C++ accesses
          // (ordered by __syncwarp) so the compiler can batch the four loads / stores of each phase.
          uint4* stg4 = reinterpret_cast<uint4*>(stg);
          if (kEpi == EPI_BF16 && use_res) {
            // residual: coalesced registers -> swizzled smem -> own row
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int rl = it * 8 + (lane >> 2);
              stg4[rl * 4 + (co_q ^ ((rl >> 1) & 3))] = rres[it];
            }
            __syncwarp();
            uint4 w4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) w4[q] = stg4[lane * 4 + (q ^ own_sw)];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              v[q * 8 + 0] += bf16_lo(w4[q].x);
              v[q * 8 + 1] += bf16_hi(w4[q].x);
              v[q * 8 + 2] += bf16_lo(w4[q].y);
              v[q * 8 + 3] += bf16_hi(w4[q].y);
              v[q * 8 + 4] += bf16_lo(w4[q].z);
              v[q * 8 + 5] += bf16_hi(w4[q].z);
              v[q * 8 + 6] += bf16_lo(w4[q].w);
              v[q * 8 + 7] += bf16_hi(w4[q].w);
            }
            __syncwarp();
            // prefetch the residual of this warp's next chunk
            if (more) load_res(col0 + 32 * EPI_PER_QUAD);
          }
          if (n_ok < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= n_ok) v[j] = 0.f;
          }
          if (kEpi == EPI_BF16 && p.rowstat_out && valid) {
            // per-row (sum, sumsq) of this 32-column chunk, for the LayerNorm folded into the consumer GEMM
            uint64_t su2 = pack_f32x2(0.f, 0.f), sq2 = su2;
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const uint64_t x2 = pack_f32x2(v[j], v[j + 1]);
              su2 = add_f32x2(su2, x2);
              sq2 = fma_f32x2(x2, x2, sq2);
            }
            float s0, s1, q0, q1;
            unpack_f32x2(su2, s0, s1);
            unpack_f32x2(sq2, q0, q1);
            p.rowstat_out[(size_t)row * p.rowstat_chunks + ((seg.out_col_off + col0) >> 5)] =
                make_float2(s0 + s1, q0 + q1);
          }
          // own row -> swizzled smem
#ifdef APTP_DBG_NOSTAGE  // kernel-tuning build: TMEM reads + epilogue math, but no staging and no stores (DESIGN 9a)
          if (v[0] == 1.2345e30f) p.abort_flag[1] = 1;
          if (p.n_tiles >= 0) continue;
#endif
#pragma unroll
          for (int q = 0; q < 4; ++q)
            stg4[lane * 4 + (q ^ own_sw)] =
                make_uint4(pack_bf16(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16(v[q * 8 + 2], v[q * 8 + 3]),
                           pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16(v[q * 8 + 6], v[q * 8 + 7]));
          if (rows_full && col0 + 32 <= seg.n_store) {
            // the staging tile IS the 64-byte-swizzled TMA box: one bulk store per chunk, nothing held in registers
            // and no per-lane store instructions queueing in the LSU
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&p.tmap_out, stg, seg.out_col_off + col0, row0_q);
              bulk_commit();
            }
            st_pending = true;
            continue;
          }
          __syncwarp();
          // coalesced side: 8 rows x 64 B per instruction
          __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + seg.out_col_off + col0 + co_q * 8;
          const bool col_ok = col0 + co_q * 8 < seg.n_store;  // n_store is a multiple of 8
          uint4 o4[4];
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rl = it * 8 + (lane >> 2);
            o4[it] = stg4[rl * 4 + (co_q ^ ((rl >> 1) & 3))];
          }
#ifdef APTP_DBG_NOSTORE  // kernel-tuning build: everything but the global stores of the bf16 path (DESIGN 9a)
          if (o4[0].x == 0x12345678u && o4[1].y == 0x9abcdef0u && o4[2].z == 0x0fedcba9u && o4[3].w == 0x87654321u)
#endif
#pragma unroll
          for (int it = 0; it < 4; ++it)
            if (co_ok[it] && col_ok) *reinterpret_cast<uint4*>(obase + (size_t)co_row[it] * p.out_ld) = o4[it];
          if constexpr (kEpi == EPI_BF16) {
            if (gn_row >= 0) {
              // column sums of the STORED (bf16-rounded) values over the 32 rows of this quadrant: 4 rows x 8 columns in
              // registers, then a fixed butterfly over the 8 lanes that share the column unit (lane bits 2..4)
              float cs[8], cq[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) cs[e] = cq[e] = 0.f;
#pragma unroll
              for (int it = 0; it < 4; ++it) {
                if (co_ok[it]) {
                  const uint32_t wds[4] = {o4[it].x, o4[it].y, o4[it].z, o4[it].w};
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float f0 = bf16_lo(wds[e]), f1 = bf16_hi(wds[e]);
                    cs[2 * e] += f0;
                    cs[2 * e + 1] += f1;
                    cq[2 * e] = fmaf(f0, f0, cq[2 * e]);
                    cq[2 * e + 1] = fmaf(f1, f1, cq[2 * e + 1]);
                  }
                }
              }
#pragma unroll
              for (int o = 4; o < 32; o <<= 1) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], o);
                  cq[e] += __shfl_xor_sync(0xffffffffu, cq[e], o);
                }
              }
              if (lane < 4 && col_ok) {
                const long long gi = gn_row + seg.out_col_off + col0 + co_q * 8;
                *reinterpret_cast<float4*>(p.gn_sum + gi) = make_float4(cs[0], cs[1], cs[2], cs[3]);
                *reinterpret_cast<float4*>(p.gn_sum + gi + 4) = make_float4(cs[4], cs[5], cs[6], cs[7]);
                *reinterpret_cast<float4*>(p.gn_sq + gi) = make_float4(cq[0], cq[1], cq[2], cq[3]);
                *reinterpret_cast<float4*>(p.gn_sq + gi + 4) = make_float4(cq[4], cq[5], cq[6], cq[7]);
              }
            }
          }
          __syncwarp();
        } else if constexpr (f32_rows) {
          uint4* stg4 = reinterpret_cast<uint4*>(stg);
          if (n_ok < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= n_ok) v[j] = 0.f;
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            // own row -> swizzled smem -> coalesced side (8 rows x 64 B per instruction). The fp32 residual was loaded
            // in the coalesced layout and is added THERE (same fp32 add, no second trip of the residual through shared
            // memory: the transposes of this epilogue moved as many shared-memory bytes as the K = 320 main loop).
#pragma unroll
            for (int q = 0; q < 4; ++q)
              stg4[lane * 4 + (q ^ own_sw)] =
                  make_uint4(__float_as_uint(v[h * 16 + q * 4 + 0]), __float_as_uint(v[h * 16 + q * 4 + 1]),
                             __float_as_uint(v[h * 16 + q * 4 + 2]), __float_as_uint(v[h * 16 + q * 4 + 3]));
            __syncwarp();
            float* obase = reinterpret_cast<float*>(p.out) + seg.out_col_off + col0 + h * 16 + co_q * 4;
            const bool col_ok = col0 + h * 16 + co_q * 4 < seg.n_store;  // n_store is a multiple of 4
            uint4 o4[4];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int rl = it * 8 + (lane >> 2);
              o4[it] = stg4[rl * 4 + (co_q ^ ((rl >> 1) & 3))];
            }
            if (use_res32) {
#pragma unroll
              for (int it = 0; it < 4; ++it) {
                o4[it].x = __float_as_uint(__uint_as_float(o4[it].x) + __uint_as_float(rres32[h][it].x));
                o4[it].y = __float_as_uint(__uint_as_float(o4[it].y) + __uint_as_float(rres32[h][it].y));
                o4[it].z = __float_as_uint(__uint_as_float(o4[it].z) + __uint_as_float(rres32[h][it].z));
                o4[it].w = __float_as_uint(__uint_as_float(o4[it].w) + __uint_as_float(rres32[h][it].w));
              }
            }
#pragma unroll
            for (int it = 0; it < 4; ++it)
              if (co_ok[it] && col_ok) *reinterpret_cast<uint4*>(obase + (size_t)co_row[it] * p.out_ld) = o4[it];
            if (gn_row >= 0) {
              // column sums of the 32 rows of this quadrant over the lane's 4 columns: 4 rows in registers, then a
              // fixed butterfly over the 8 lanes that share the column unit (lane bits 2..4)
              float cs[4] = {0.f, 0.f, 0.f, 0.f}, cq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int it = 0; it < 4; ++it) {
                if (co_ok[it]) {
                  const float f0 = __uint_as_float(o4[it].x), f1 = __uint_as_float(o4[it].y);
                  const float f2 = __uint_as_float(o4[it].z), f3 = __uint_as_float(o4[it].w);
                  cs[0] += f0; cs[1] += f1; cs[2] += f2; cs[3] += f3;
                  cq[0] = fmaf(f0, f0, cq[0]); cq[1] = fmaf(f1, f1, cq[1]);
                  cq[2] = fmaf(f2, f2, cq[2]); cq[3] = fmaf(f3, f3, cq[3]);
                }
              }
#pragma unroll
              for (int o = 4; o < 32; o <<= 1) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], o);
                  cq[e] += __shfl_xor_sync(0xffffffffu, cq[e], o);
                }
              }
              if (lane < 4 && col_ok) {
                const long long gi = gn_row + seg.out_col_off + col0 + h * 16 + co_q * 4;
                *reinterpret_cast<float4*>(p.gn_sum + gi) = make_float4(cs[0], cs[1], cs[2], cs[3]);
                *reinterpret_cast<float4*>(p.gn_sq + gi) = make_float4(cq[0], cq[1], cq[2], cq[3]);
              }
            }
            __syncwarp();
          }
          if (use_res32 && more) load_res32(col0 + 32 * EPI_PER_QUAD);  // after the stores: `residual` may alias `out`
        } else if (valid) {
          if (n_ok < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= n_ok) v[j] = 0.f;
          }
          {  // fp32 NCHW: out[(sample*out_ld + col) * rows_per_sample + pixel]
            float* op = reinterpret_cast<float*>(p.out);
            const int pix = row - sample * p.rows_per_sample;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < n_ok) op[((size_t)sample * p.out_ld + col0 + j) * p.rows_per_sample + pix] = v[j];
          }
        }
#ifdef APTP_GEMM_TRACE
        _tr_st += clock64() - _c2;
#endif
      }
      if (!released) release_acc();  // no chunk of this tile fell to this warp
#ifdef APTP_GEMM_TRACE
      _tr_busy += clock64() - _e1;
      _tr_tiles += 1;
#endif
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) bulk_wait0();  // outstanding bulk stores (their shared-memory source dies with the CTA)
#ifdef APTP_GEMM_TRACE
    if (lane == 0 && ew < 2) {
      g_gemm_trace[blockIdx.x][6 + 3 * ew] += _tr_tfull;
      g_gemm_trace[blockIdx.x][7 + 3 * ew] += _tr_busy;
      g_gemm_trace[blockIdx.x][8 + 3 * ew] += _tr_tiles;
      if (ew == 0) {
        g_gemm_trace[blockIdx.x][12] += _tr_ld;
        g_gemm_trace[blockIdx.x][13] += _tr_math;
        g_gemm_trace[blockIdx.x][14] += _tr_st;
      }
    }
#endif
  }

#ifdef APTP_GEMM_TRACE
  if (warp == 4 && lane == 0) g_gemm_trace[blockIdx.x][5] += clock64() - _t0_epi;
#endif
  tc_fence_before();
  cluster_sync_all();  // the peer may still multicast into this CTA's smem / arrive on its barriers until here
  if (warp == 1) {
    tc_fence_after();
    if constexpr (k2Sm) tmem_dealloc_2sm(*tmem_slot, TMEM_COLS);
    else tmem_dealloc(*tmem_slot, TMEM_COLS);
  }
}

#ifdef APTP_GEMM_TRACE
}  // namespace aptp
extern "C" int aptp_debug_gemm_trace(long long* host_out, int reset) {  // [512][16]
  if (host_out && cudaMemcpyFromSymbol(host_out, aptp::g_gemm_trace, sizeof(long long) * 512 * 16) != cudaSuccess) return -1;
  if (reset) {
    static long long zeros[512 * 16];
    if (cudaMemcpyToSymbol(aptp::g_gemm_trace, zeros, sizeof(zeros)) != cudaSuccess) return -1;
  }
  return 0;
}
namespace aptp {
#endif
static int g_gemm_smem_set = 0;
static int g_gemm_max_clusters = 0;
static int g_gemm_2sm = 1;
// Measured on B200 (tools/gemm_bench.py, same box): 3x3 convs +8..17 %, K = N = 1280 linear +13 %, 8192^3 +8 % with the
// 2-SM scheme, but the K = 320 / 640 projections LOSE 10..25 % (their tiles are 5-10 K steps long and every tile
// hand-off crosses the CTA pair), so short reductions keep the two independent M = 128 MMAs.
static int g_gemm_2sm_mink = 1280;
static int g_conv_halo = 1;  // APTP_CONV_HALO=0: nine shifted boxes per K chunk (round-1 scheme) for A/B runs

}  // namespace aptp

using namespace aptp;

static int gemm_max_clusters() {
  if (!g_gemm_smem_set) {
    const void* fns[8] = {(const void*)grouped_gemm_kernel<EPI_BF16, false>, (const void*)grouped_gemm_kernel<EPI_GEGLU, false>,
                          (const void*)grouped_gemm_kernel<EPI_F32, false>,  (const void*)grouped_gemm_kernel<EPI_NCHW, false>,
                          (const void*)grouped_gemm_kernel<EPI_BF16, true>,  (const void*)grouped_gemm_kernel<EPI_GEGLU, true>,
                          (const void*)grouped_gemm_kernel<EPI_F32, true>,   (const void*)grouped_gemm_kernel<EPI_NCHW, true>};
    for (int i = 0; i < 8; ++i)
      if (cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return 0;
    // APTP_GEMM_1SM=1: the round-1 scheme (two M = 128 MMAs per pair over a multicast B tile) everywhere, for A/B runs;
    // APTP_GEMM_2SM_MINK: shortest reduction length (K, times 9 for the convs) that takes the 2-SM scheme
    const char* e = getenv("APTP_GEMM_1SM");
    g_gemm_2sm = !(e && e[0] == '1');
    const char* hl = getenv("APTP_CONV_HALO");
    if (hl && hl[0] == '0') g_conv_halo = 0;
    const char* mk = getenv("APTP_GEMM_2SM_MINK");
    if (mk && atoi(mk) > 0) g_gemm_2sm_mink = atoi(mk);
    g_gemm_smem_set = 1;
  }
  if (!g_gemm_max_clusters) {
    // CTA pairs must land on one GPC: the number of co-resident pairs can be below sm_count()/2
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(sm_count() & ~1, 1, 1);
    cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
    cfg.dynamicSmemBytes = 227 * 1024;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, grouped_gemm_kernel<EPI_BF16, true>, &cfg) != cudaSuccess || n <= 0) return 0;
    g_gemm_max_clusters = n;
  }
  return g_gemm_max_clusters;
}

extern "C" int aptp_gemm_max_pairs(void) { return gemm_max_clusters(); }

extern "C" int aptp_grouped_gemm_fwd(const aptp_gemm_args* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  APTP_REQUIRE(a != nullptr, "aptp_grouped_gemm_fwd: null args");
  APTP_REQUIRE(a->a && a->w && a->out && a->segs && a->tiles, "aptp_grouped_gemm_fwd: null pointer");
  if (a->n_tiles == 0) return APTP_OK;
  APTP_REQUIRE(a->n_tiles % 2 == 0, "aptp_grouped_gemm_fwd: tiles must come in pairs (n_tiles=%d is odd)", a->n_tiles);
  APTP_REQUIRE(a->bn >= 32 && a->bn <= 256 && a->bn % 32 == 0, "aptp_grouped_gemm_fwd: bn=%d must be a multiple of 32 in [32,256]", a->bn);
  APTP_REQUIRE(a->a_ld % 8 == 0 && a->w_ld % 8 == 0, "aptp_grouped_gemm_fwd: a_ld/w_ld must be multiples of 8 (16-byte rows)");
  APTP_REQUIRE(a->out_mode == APTP_OUT_F32_NCHW || a->out_ld % 8 == 0, "aptp_grouped_gemm_fwd: out_ld must be a multiple of 8");
  APTP_REQUIRE((reinterpret_cast<uintptr_t>(a->a) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->w) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(a->out) & 15) == 0,
               "aptp_grouped_gemm_fwd: operands must be 16-byte aligned");
  APTP_REQUIRE(a->rows_per_sample > 0, "aptp_grouped_gemm_fwd: rows_per_sample must be > 0");
  if (a->flags & APTP_EPI_RES_F32)
    APTP_REQUIRE(a->residual != nullptr && a->out_mode == APTP_OUT_F32 && a->res_ld % 4 == 0 &&
                     (reinterpret_cast<uintptr_t>(a->residual) & 15) == 0,
                 "aptp_grouped_gemm_fwd: APTP_EPI_RES_F32 needs an fp32 residual (16-byte aligned rows) and APTP_OUT_F32");
  else
    APTP_REQUIRE(a->residual == nullptr || (a->out_mode == APTP_OUT_BF16 && a->res_ld % 8 == 0),
                 "aptp_grouped_gemm_fwd: a bf16 residual needs a bf16 output and res_ld %% 8 == 0");
  APTP_REQUIRE(a->a_rows < (1ll << 31), "aptp_grouped_gemm_fwd: too many rows");
  if (a->flags & APTP_EPI_GN_STATS) {
    APTP_REQUIRE(a->gn_stats && a->gn_stats_sq && (a->out_mode == APTP_OUT_F32 || a->out_mode == APTP_OUT_BF16) &&
                     !(a->flags & APTP_EPI_GEGLU),
                 "aptp_grouped_gemm_fwd: APTP_EPI_GN_STATS needs both partial planes and a row output (fp32 or bf16)");
    APTP_REQUIRE(a->rows_per_sample % 128 == 0 && a->gn_blocks == a->rows_per_sample / 32 && a->gn_ld % 4 == 0,
                 "aptp_grouped_gemm_fwd: APTP_EPI_GN_STATS needs rows_per_sample %% 128 == 0, gn_blocks = rows_per_sample / 32");
    APTP_REQUIRE(a->a_mode == APTP_A_LINEAR || a->bb == 1, "aptp_grouped_gemm_fwd: APTP_EPI_GN_STATS needs conv boxes inside one image");
    APTP_REQUIRE((reinterpret_cast<uintptr_t>(a->gn_stats) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->gn_stats_sq) & 15) == 0,
                 "aptp_grouped_gemm_fwd: partial planes must be 16-byte aligned");
  }
  if (a->flags & APTP_EPI_LN_FOLD) {
    APTP_REQUIRE(a->ln_colsum && a->ln_rowstats && a->bias && (reinterpret_cast<uintptr_t>(a->ln_rowstats) & 7) == 0,
                 "aptp_grouped_gemm_fwd: APTP_EPI_LN_FOLD needs ln_colsum, ln_rowstats and bias (= W @ beta + layer bias)");
    APTP_REQUIRE(a->a_mode == APTP_A_LINEAR, "aptp_grouped_gemm_fwd: APTP_EPI_LN_FOLD applies to linear layers");
  }
  if (a->rowstat_out) {
    APTP_REQUIRE(a->out_mode == APTP_OUT_BF16 && !(a->flags & APTP_EPI_GEGLU) && a->rowstat_chunks > 0 && a->bn % 32 == 0,
                 "aptp_grouped_gemm_fwd: rowstat_out needs a plain bf16 output");
  }
  if (a->flags & APTP_EPI_GEGLU) {
    APTP_REQUIRE(a->bn % 64 == 0, "aptp_grouped_gemm_fwd: GEGLU needs bn %% 64 == 0");
    APTP_REQUIRE(a->out_mode == APTP_OUT_BF16 && !a->residual && !a->rowvec && !a->border_tab && !(a->flags & APTP_EPI_SILU),
                 "aptp_grouped_gemm_fwd: the GEGLU epilogue takes bias and gate only and writes bf16");
  }

  GemmParams p;
  memset(&p, 0, sizeof(p));
  int Ho = 1, Wo = 1;
  APTP_REQUIRE(gemm_max_clusters() > 0, "aptp_grouped_gemm_fwd: no CTA pair fits on this device");
  // (the opt-in A-stationary layout exists in the 1-SM scheme only)
  const bool two_sm = g_gemm_2sm && a->a_stat_chunks <= 0 && (a->a_mode == APTP_A_LINEAR ? 1 : 9) * a->a_k >= g_gemm_2sm_mink;
  // halo tile instead of nine shifted boxes: 2-SM stride-1 3x3 convs whose schedule uses 8 x 16 pixel boxes
  const bool halo = two_sm && g_conv_halo && a->a_mode == APTP_A_CONV3X3 && a->bw == 8 && a->bh == 16 && a->bb == 1;
  if (a->a_mode == APTP_A_LINEAR) {
    uint64_t dims[2] = {(uint64_t)a->a_k, (uint64_t)a->a_rows};
    uint64_t strides[1] = {(uint64_t)a->a_ld * 2};
    uint32_t box[2] = {BK, BM};
    int rc = make_tmap_bf16(&p.tmap_a, a->a, 2, dims, strides, box);
    if (rc) return rc;
  } else if (a->a_mode == APTP_A_CONV3X3) {
    APTP_REQUIRE(a->bw * a->bh * a->bb == BM, "aptp_grouped_gemm_fwd: conv box %dx%dx%d != 128 pixels", a->bw, a->bh, a->bb);
    Ho = a->H;
    Wo = a->W;
    APTP_REQUIRE(Wo % a->bw == 0 && Ho % a->bh == 0, "aptp_grouped_gemm_fwd: box does not tile the image");
    uint64_t dims[4] = {(uint64_t)a->a_k, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->batch};
    uint64_t strides[3] = {(uint64_t)a->a_ld * 2, (uint64_t)a->W * a->a_ld * 2, (uint64_t)a->H * a->W * a->a_ld * 2};
    uint32_t box[4] = {BK, (uint32_t)a->bw, (uint32_t)a->bh, (uint32_t)a->bb};
    if (halo) {
      box[1] = HALO_W;
      box[2] = HALO_H;
    }
    int rc = make_tmap_bf16(&p.tmap_a, a->a, 4, dims, strides, box);
    if (rc) return rc;
  } else if (a->a_mode == APTP_A_CONV3X3_S2) {
    APTP_REQUIRE(a->bw * a->bh * a->bb == BM, "aptp_grouped_gemm_fwd: conv box != 128 pixels");
    APTP_REQUIRE(a->H % 2 == 0 && a->W % 2 == 0, "aptp_grouped_gemm_fwd: stride-2 conv needs even H, W");
    APTP_REQUIRE(a->a_k == a->a_ld && a->k_tap_pitch == a->a_ld, "aptp_grouped_gemm_fwd: stride-2 conv needs a_k == a_ld == k_tap_pitch");
    Ho = a->H / 2;
    Wo = a->W / 2;
    APTP_REQUIRE(Wo % a->bw == 0 && Ho % a->bh == 0, "aptp_grouped_gemm_fwd: box does not tile the image");
    // view [b][H/2][2][W/2][2][C] as dims (fastest first): (px*C + c), W/2, py, H/2, b
    uint64_t dims[5] = {(uint64_t)2 * a->a_ld, (uint64_t)Wo, 2, (uint64_t)Ho, (uint64_t)a->batch};
    uint64_t strides[4] = {(uint64_t)2 * a->a_ld * 2, (uint64_t)a->W * a->a_ld * 2,
                           (uint64_t)2 * a->W * a->a_ld * 2, (uint64_t)a->H * a->W * a->a_ld * 2};
    uint32_t box[5] = {BK, (uint32_t)a->bw, 1, (uint32_t)a->bh, (uint32_t)a->bb};
    int rc = make_tmap_bf16(&p.tmap_a, a->a, 5, dims, strides, box);
    if (rc) return rc;
  } else {
    APTP_REQUIRE(false, "aptp_grouped_gemm_fwd: bad a_mode %d", a->a_mode);
  }
  {
    uint64_t dims[2] = {(uint64_t)a->w_ld, (uint64_t)a->w_rows};
    uint64_t strides[1] = {(uint64_t)a->w_ld * 2};
    uint32_t box[2] = {BK, (uint32_t)a->bn / 2};  // each CTA of a pair loads (and multicasts) half of the weight tile
    int rc = make_tmap_bf16(&p.tmap_b, a->w, 2, dims, strides, box);
    if (rc) return rc;
  }
  p.k2_chunks = 0;
  if (a->a2 != nullptr) {
    if (!halo) {
      set_error("aptp_grouped_gemm_fwd: the second operand pair (a2 / w2) needs the halo-tile conv scheme");
      return APTP_ERR_UNSUPPORTED;
    }
    APTP_REQUIRE(a->w2 && a->a2_k > 0 && a->a2_k % 8 == 0 && a->a2_ld % 8 == 0 && a->w2_ld % 8 == 0 && a->w2_rows > 0 &&
                     !(a->flags & APTP_EPI_GEGLU),
                 "aptp_grouped_gemm_fwd: bad second operand pair");
    uint64_t dims[4] = {(uint64_t)a->a2_k, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->batch};
    uint64_t strides[3] = {(uint64_t)a->a2_ld * 2, (uint64_t)a->W * a->a2_ld * 2, (uint64_t)a->H * a->W * a->a2_ld * 2};
    uint32_t box[4] = {BK, 8, 16, 1};
    int rc = make_tmap_bf16(&p.tmap_a2, a->a2, 4, dims, strides, box);
    if (rc) return rc;
    uint64_t wdims[2] = {(uint64_t)a->w2_ld, (uint64_t)a->w2_rows};
    uint64_t wstrides[1] = {(uint64_t)a->w2_ld * 2};
    uint32_t wbox[2] = {BK, (uint32_t)a->bn / 2};
    rc = make_tmap_bf16(&p.tmap_b2, a->w2, 2, wdims, wstrides, wbox);
    if (rc) return rc;
    p.k2_chunks = (a->a2_k + BK - 1) / BK;
  }
  p.segs = a->segs;
  p.tiles = a->tiles;
  p.n_tiles = a->n_tiles;
  p.n_segs = a->n_segs;
  p.a_mode = a->a_mode;
  p.batch = a->batch;
  p.Ho = Ho;
  p.Wo = Wo;
  p.bn = a->bn;
  p.bw = a->a_mode == APTP_A_LINEAR ? BM : a->bw;
  p.bh = a->a_mode == APTP_A_LINEAR ? 1 : a->bh;
  p.bb = a->a_mode == APTP_A_LINEAR ? 1 : a->bb;
  APTP_REQUIRE((p.bw & (p.bw - 1)) == 0 && (p.bh & (p.bh - 1)) == 0, "aptp_grouped_gemm_fwd: box extents must be powers of two");
  p.lbw = 0;
  while ((1 << p.lbw) < p.bw) ++p.lbw;
  p.lbh = 0;
  while ((1 << p.lbh) < p.bh) ++p.lbh;
  p.k_tap_pitch = a->k_tap_pitch;
  p.out = a->out;
  p.out_ld = a->out_ld;
  p.out_mode = a->out_mode;
  p.out_tma = 0;
  {
    static int tma_store = -1;  // APTP_GEMM_TMA_STORE=0: per-lane stores everywhere (A/B runs)
    if (tma_store < 0) {
      const char* e = getenv("APTP_GEMM_TMA_STORE");
      tma_store = !(e && e[0] == '0');
    }
    if (tma_store && a->a_mode == APTP_A_LINEAR && a->out_mode == APTP_OUT_BF16 && !(a->flags & APTP_EPI_GN_STATS) &&
        (reinterpret_cast<uintptr_t>(a->out) & 15) == 0) {
      const uint64_t out_cols = (uint64_t)a->out_ld;  // columns addressable in a row (segments write disjoint column ranges)
      int rc = make_tmap_store64(&p.tmap_out, a->out, false, out_cols, (uint64_t)a->a_rows, (uint64_t)a->out_ld * 2);
      if (rc) return rc;
      p.out_tma = 1;
    }
  }
  p.bias = a->bias;
  p.rowvec = a->rowvec;
  p.rowvec_ld = a->rowvec_ld;
  p.rows_per_sample = a->rows_per_sample;
  p.residual = a->residual;
  p.res_ld = a->res_ld;
  p.gate = a->gate;
  p.gate_ld = a->gate_ld;
  p.gate_group = a->gate_group > 0 ? a->gate_group : 1;
  p.border_tab = a->border_tab;
  p.tab_ld = a->tab_ld;
  p.flags = a->flags;
  p.ln_colsum = a->ln_colsum;
  p.ln_rowstats = reinterpret_cast<const float2*>(a->ln_rowstats);
  p.rowstat_out = reinterpret_cast<float2*>(a->rowstat_out);
  p.rowstat_chunks = a->rowstat_chunks;
  const bool gn = (a->flags & APTP_EPI_GN_STATS) != 0;
  p.gn_sum = gn ? a->gn_stats : nullptr;
  p.gn_sq = gn ? a->gn_stats_sq : nullptr;
  p.gn_ld = a->gn_ld;
  p.gn_blocks = a->gn_blocks;
  p.abort_flag = device_abort_flag();
  APTP_REQUIRE(p.abort_flag != nullptr, "aptp_grouped_gemm_fwd: could not allocate abort flag");

  p.a_stat = 0;
  if (a->a_stat_chunks > 0) {
    APTP_REQUIRE(a->a_mode == APTP_A_LINEAR && a->a_stat_chunks <= A_STAT_MAX_CHUNKS,
                 "aptp_grouped_gemm_fwd: A-stationary mode needs a linear layer with at most %d K chunks", A_STAT_MAX_CHUNKS);
    p.a_stat = a->a_stat_chunks;
  }
  const int stage_bytes = ((p.a_stat || halo) ? 0 : A_STAGE_BYTES) + a->bn * (two_sm ? 64 : 128);
  p.halo = 0;
  if (halo) {  // 2 halo slots, a third one when the weight ring still gets 8 stages
    p.halo = 2;
    const int b8 = 8 * stage_bytes;
    if (225 * 1024 - 1024 - 512 - STG_BYTES - SBIAS_BYTES - SSEG_BYTES - STILE_BYTES - 3 * HALO_BYTES >= b8) p.halo = 3;
  }
  const int a_region = p.halo ? p.halo * HALO_BYTES : p.a_stat * A_STAGE_BYTES;
  const int budget = 225 * 1024 - 1024 /*align slack*/ - 512 /*barriers*/ - STG_BYTES /*epilogue staging*/ - SBIAS_BYTES -
                     SSEG_BYTES - STILE_BYTES - a_region;
  int stages = budget / stage_bytes;
  if (stages > 8) stages = 8;
  APTP_REQUIRE(stages >= 2, "aptp_grouped_gemm_fwd: tile too large for shared memory");
  p.stages = stages;
  const size_t smem_bytes = (size_t)a_region + (size_t)stages * stage_bytes + STG_BYTES + SBIAS_BYTES +
                            SSEG_BYTES + STILE_BYTES + 1024 + 512;
  const int n_pairs = a->n_tiles / 2;
  int grid = 2 * (n_pairs < g_gemm_max_clusters ? n_pairs : g_gemm_max_clusters);
  if (p.a_stat) {  // the tile list was laid out for exactly a_stat_pairs CTA pairs (entry c + j * pairs belongs to pair c)
    APTP_REQUIRE(a->a_stat_pairs > 0 && a->a_stat_pairs <= g_gemm_max_clusters && n_pairs % a->a_stat_pairs == 0,
                 "aptp_grouped_gemm_fwd: A-stationary tile list needs 0 < a_stat_pairs <= %d dividing the pair count", g_gemm_max_clusters);
    grid = 2 * a->a_stat_pairs;
  }
#define APTP_LAUNCH_GEMM(EPI)                                                                  \
  do {                                                                                         \
    if (two_sm) APTP_CUDA_CHECK(launch_pdl(grouped_gemm_kernel<EPI, true>, dim3(grid), dim3(GEMM_THREADS), smem_bytes, stream, p)); \
    else APTP_CUDA_CHECK(launch_pdl(grouped_gemm_kernel<EPI, false>, dim3(grid), dim3(GEMM_THREADS), smem_bytes, stream, p));       \
  } while (0)
  if (a->flags & APTP_EPI_GEGLU) APTP_LAUNCH_GEMM(EPI_GEGLU);
  else if (a->out_mode == APTP_OUT_BF16) APTP_LAUNCH_GEMM(EPI_BF16);
  else if (a->out_mode == APTP_OUT_F32) APTP_LAUNCH_GEMM(EPI_F32);
  else APTP_LAUNCH_GEMM(EPI_NCHW);
#undef APTP_LAUNCH_GEMM
  APTP_CUDA_CHECK(cudaGetLastError());
  return APTP_OK;
}
